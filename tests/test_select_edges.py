"""Edges of the device-side allele selection (`mmlst_select_dev`, csrc/select.cu) at the shape of a real MLST database, against a plain Python
restatement of metamlst.py:133-220 written here (`select_reference`: Python ints and floats, `round(x, 1)` on every hit allele, the oracle's
`select_alleles`, the --nloci gate, H5 order, column layout and chunk list):

- loci longer than the kernel's register window of SEL_R x 256 = 1024 allele rows (the remainder loops of all three passes): winners beyond
  row 1024, rounded-average ties across the window edge, the locus maximum hit count held only by a remainder row, and the MMLST_SELECT_CONSUME
  reset of remainder rows, with the rows grouped by locus (no row list) and interleaved (row list);
- 32 to about 5000 loci and 1 to 4096 species: the CTA-wide finalizer (the only one past 32 loci or species), dynamic shared memory past the
  48 KB every kernel starts with, the largest index the device accepts and the MMLST_E_RANGE refusal of the next one;
- rounding at hit counts up to 2^32 - 1, sums up to about 2^50, negative averages and every penalty, on exact binary ties and on quotients
  within one ulp of a tie, each paired with a rival that wins or loses if the rounding is one tenth off;
- the --nloci gate for 1-100 genes at every detected count, at, below and above the threshold, the "Database is broken" bit and
  MMLST_SELECT_LOCAL;
- every output: header, chosen rows / species / first records / columns / DB offsets, the chunk list under three chunk rules, chunk-list
  overflow, the counters, and a second call on new tables after a consuming one;
- one synthetic DB of that shape (34 species, two loci of more than 1024 alleles) end to end through DevicePipeline and mmlst_sample.

Every case asserts the regime it targets from mirrors of the kernel's constants.  Needs a B200 except for the host checks: `pytest -m gpu`."""
import ctypes as C
import math
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

from metamlst_b200 import api, native
from oracle import mlst_oracle as orc

gpu = pytest.mark.gpu

# ------------------------------------------------------------------------------------------------ mirrors of the kernel's constants
SEL_THREADS, SEL_R = 256, 4
WINDOW = SEL_R * SEL_THREADS   # allele rows of a locus held in registers; the rest are read from memory in a second loop of every pass
DEFAULT_SMEM = 48 * 1024       # dynamic shared memory a kernel may use without opting in (less its static part)
NO_IDX = 0xFFFFFFFF
SENT = 0x5A5A5A5A              # what the driver fills every output with: words the kernel must not write keep it
CONSUME, SCRATCH_CLEAN, LOCAL = native.SELECT_CONSUME, native.SELECT_SCRATCH_CLEAN, native.SELECT_LOCAL


def smem_bytes(n_loci, n_species):
    """Mirror of select_smem_bytes (csrc/select.cu): dynamic shared memory of one selection launch."""
    return max(4 * (11 * n_loci + 1 + 4 * n_species) + 16, 800)


def warp_finalizer(n_loci, n_species, warp):
    """Mirror of the finalizer choice in sel_locus: the one-warp form only when switched on and n_loci, n_species <= 32."""
    return bool(warp) and n_loci <= 32 and n_species <= 32


# ------------------------------------------------------------------------------------------------ tables
class Tables:
    """One selection problem: per allele row its locus, allele number, score tables (sum of AS, hits, first passing record), pileup record
    count, BAM LN and DB sequence length; per locus its species; per species the rows of `genes`; the two read counters."""

    def __init__(self, locus_of, allele_num, sol, gdb, sum_as, n_hit, first_idx, nrec=None, ref_len=None, db_len=None, counters=(0, 0), seed=0):
        rng = np.random.default_rng(seed)
        n = len(locus_of)
        self.locus_of = np.asarray(locus_of, np.uint32)
        self.allele_num = np.asarray(allele_num, np.uint32)
        self.sol = np.asarray(sol, np.uint32)
        self.gdb = np.asarray(gdb, np.uint32)
        self.sum_as = np.asarray(sum_as, np.int64)
        self.n_hit = np.asarray(n_hit, np.uint32)
        self.first_idx = np.asarray(first_idx, np.uint32)
        self.nrec = np.asarray(nrec if nrec is not None else rng.integers(0, 3000, n), np.int64)
        self.ref_len = np.asarray(ref_len if ref_len is not None else rng.integers(1, 1500, n), np.uint32)
        self.db_len = np.asarray(db_len if db_len is not None else self.ref_len.astype(np.int64) + rng.integers(0, 40, n), np.int64)
        self.counters = tuple(int(c) for c in counters)
        self.n_ref, self.n_loci, self.n_species = n, len(self.sol), len(self.gdb)
        assert self.first_idx[self.n_hit == 0].tolist() == [NO_IDX] * int((self.n_hit == 0).sum()) and not self.sum_as[self.n_hit == 0].any()
        key = self.locus_of.astype(np.int64) << 32 | self.allele_num
        assert np.unique(key).shape[0] == n, "allele numbers must be unique inside a locus"

    # derived tables, as the kernel receives them
    @property
    def contig_start(self):   # pileup-stream record range of every row; starts past 0
        return np.concatenate([[0], np.cumsum(self.nrec)]).astype(np.uint64) + np.uint64(1000)

    @property
    def db_off(self):         # DB sequence offsets past 2^32
        return np.concatenate([[0], np.cumsum(self.db_len)]).astype(np.uint64) + np.uint64(3 << 32)

    @property
    def order(self):          # allele rows grouped by locus, ascending row inside a locus
        return np.argsort(self.locus_of, kind="stable").astype(np.uint32)

    @property
    def grouped(self):
        return bool(np.array_equal(self.order, np.arange(self.n_ref, dtype=np.uint32)))

    @property
    def locus_start(self):
        return np.searchsorted(self.locus_of[self.order], np.arange(self.n_loci + 1)).astype(np.uint32)

    def pos_in_locus(self):
        """Index of every row inside its locus's row list: >= WINDOW = read by the remainder loops."""
        o = self.order
        pos = np.zeros(self.n_ref, np.int64)
        pos[o] = np.arange(self.n_ref) - self.locus_start[self.locus_of[o]]
        return pos

    def permuted(self, src):
        return Tables(self.locus_of[src], self.allele_num[src], self.sol, self.gdb, self.sum_as[src], self.n_hit[src], self.first_idx[src],
                      self.nrec[src], self.ref_len[src], self.db_len[src], self.counters)

    def interleaved(self, rng):
        """The same loci with their rows interleaved (the kernel needs the row list); every locus keeps the order of its own rows."""
        labels = rng.permutation(self.locus_of)
        src = np.empty(self.n_ref, np.int64)
        src[np.argsort(labels, kind="stable")] = self.order
        t = self.permuted(src)
        assert not t.grouped
        return t

    def with_scores(self, sum_as, n_hit, first_idx, counters):
        t = Tables(self.locus_of, self.allele_num, self.sol, self.gdb, sum_as, n_hit, first_idx, self.nrec, self.ref_len, self.db_len, counters)
        return t


def unique_firsts(rng, n_hit):
    f = np.full(n_hit.shape[0], NO_IDX, np.uint32)
    h = np.nonzero(n_hit)[0]
    f[h] = rng.choice(50_000_000, h.shape[0], replace=False).astype(np.uint32)
    return f


# ------------------------------------------------------------------------------------------------ reference
def select_reference(tb, penalty=100, nloci=100, flags=0, chunk_records=512, max_chunks=None):
    """metamlst.py:133-151 (maxLen, penalty, round(avg, 1) per hit allele), :244 (lowest int(allele) among the best, oracle's select_alleles),
    :184-206 (gate; tot < det = "Database is broken"), H5 order (species, then loci, by first passing record), then the column layout
    (exclusive prefix of BAM LN), DB offsets and the chunk list (ceil(records / chunk_records) chunks per chosen locus, at least one)."""
    rows_of = {}
    for t in np.nonzero(tb.n_hit)[0].tolist():
        rows_of.setdefault(int(tb.locus_of[t]), []).append(t)
    chosen, lfirst = {}, {}
    for l, rows in rows_of.items():
        maxLen = max(int(tb.n_hit[t]) for t in rows)
        info, row_of = {}, {}
        for t in rows:
            geneLen, localScore = int(tb.n_hit[t]), int(tb.sum_as[t])
            if geneLen != maxLen:
                localScore = localScore - (maxLen - geneLen) * penalty
            a = str(int(tb.allele_num[t]))
            info[a] = (localScore, geneLen, round(float(localScore) / float(geneLen), 1))
            row_of[a] = t
        ((_g, a),) = orc.select_alleles({l: info})
        chosen[l] = row_of[a]
        lfirst[l] = min(int(tb.first_idx[t]) for t in rows)
    det, sp_first = {}, {}
    for l in chosen:
        sp = int(tb.sol[l])
        det[sp] = det.get(sp, 0) + 1
        sp_first[sp] = min(sp_first.get(sp, NO_IDX), lfirst[l])
    err, passed = 0, set()
    for sp, d in det.items():
        tot = int(tb.gdb[sp])
        if flags & LOCAL:
            passed.add(sp)
        elif tot < d:
            err |= 1
        elif int((float(d) / float(tot)) * 100) >= nloci:
            passed.add(sp)
    kept = sorted((l for l in chosen if int(tb.sol[l]) in passed), key=lambda l: (sp_first[int(tb.sol[l])], lfirst[l], l))
    tid = [chosen[l] for l in kept]
    cs, dbo = tb.contig_start, tb.db_off
    col_off = [0]
    for t in tid:
        col_off.append(col_off[-1] + int(tb.ref_len[t]))
    nrec = [int(cs[t + 1]) - int(cs[t]) for t in tid]
    cr = chunk_records or int(native.lib().mmlst_chunk_records(sum(nrec)))
    chunks = []
    for i, t in enumerate(tid):
        q0, k = int(cs[t]), max(1, -(-nrec[i] // cr))
        for j in range(k):
            chunks.append((q0 + j * cr, min(q0 + (j + 1) * cr, q0 + nrec[i]), col_off[i], int(tb.ref_len[t]), 0, i, k, 0))
    if max_chunks is not None and len(chunks) > max_chunks:
        err |= 2
    n_listed = len(chunks) if max_chunks is None else min(len(chunks), max_chunks)
    return {"n": len(tid), "n_chunks_needed": len(chunks), "header": [len(tid), n_listed, col_off[-1], err, cr], "tid": tid,
            "species": [int(tb.sol[l]) for l in kept], "first": [lfirst[l] for l in kept], "col_off": col_off,
            "db_start": [int(dbo[t]) for t in tid], "chunks": chunks[:n_listed], "chosen_locus": dict(chosen)}


# ------------------------------------------------------------------------------------------------ driver
class Selector:
    """mmlst_select_dev over device copies of `tb`, every argument and output exposed.  The tables stay resident, so a call can be repeated
    (another gate, chunk rule, flag set) or follow a consuming one; `load` puts new score tables and counters in the same buffers."""

    def __init__(self, tb, row_list=None):
        dev = torch.device("cuda:0")
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.tb = tb
        self.sum_as, self.n_hit, self.first_idx = d(tb.sum_as), d(tb.n_hit.view(np.int32)), d(tb.first_idx.view(np.int32))
        use_rows = (not tb.grouped) if row_list is None else row_list
        self.rows = d(tb.order.view(np.int32)) if use_rows else None
        self.start, self.allele = d(tb.locus_start.view(np.int32)), d(tb.allele_num.view(np.int32))
        self.sol, self.gdb = d(tb.sol.view(np.int32)), d(tb.gdb.view(np.int32))
        self.cs, self.rl, self.dbo = d(tb.contig_start.view(np.int64)), d(tb.ref_len.view(np.int32)), d(tb.db_off.view(np.int64))
        self.counters = d(np.asarray(tb.counters, np.uint64).view(np.int64))
        self.scratch = torch.zeros(tb.n_loci * 12 + 64, dtype=torch.uint8, device=dev)
        self.dev = dev

    def load(self, tb):
        self.tb = tb
        for dst, src in ((self.sum_as, tb.sum_as), (self.n_hit, tb.n_hit.view(np.int32)), (self.first_idx, tb.first_idx.view(np.int32)),
                         (self.counters, np.asarray(tb.counters, np.uint64).view(np.int64))):
            dst.copy_(torch.from_numpy(np.ascontiguousarray(src)))

    def call(self, penalty=100, nloci=100, flags=0, chunk_records=512, max_chunks=None, warp=0, want_first=True, want_counters=True,
             n_loci=None, n_species=None):
        """-> rc, outputs (numpy).  n_loci / n_species override the index shape (range checks only)."""
        tb, nl = self.tb, self.tb.n_loci
        if max_chunks is None:
            max_chunks = nl + int(tb.nrec.sum()) // 512 + 8
        out = lambda n, dt=torch.int32: torch.full((n,), SENT, dtype=dt, device=self.dev)
        hdr, tid, sp, col, first = out(16), out(nl), out(nl), out(nl + 1), out(nl)
        dbs = torch.full((nl,), SENT | (SENT << 32), dtype=torch.int64, device=self.dev)
        chunks = out(8 * (max_chunks + 4))
        lib = native.lib()
        prev = lib.mmlst_set_select_warp_finalize(int(warp))
        try:
            rc = lib.mmlst_select_dev(native.ptr(self.sum_as), native.ptr(self.n_hit), native.ptr(self.first_idx), native.ptr(self.rows),
                                      native.ptr(self.start), native.ptr(self.allele), tb.n_ref, native.ptr(self.sol), native.ptr(self.gdb),
                                      nl if n_loci is None else n_loci, tb.n_species if n_species is None else n_species, int(penalty), int(nloci),
                                      native.ptr(self.cs), native.ptr(self.rl), native.ptr(self.dbo), int(chunk_records), native.ptr(self.scratch),
                                      int(self.scratch.shape[0]), native.ptr(hdr), native.ptr(tid), native.ptr(sp), native.ptr(col), native.ptr(dbs),
                                      native.ptr(chunks), int(max_chunks), int(flags), native.ptr(self.counters) if want_counters else 0,
                                      native.ptr(first) if want_first else 0, torch.cuda.current_stream(self.dev).cuda_stream)
        finally:
            assert lib.mmlst_set_select_warp_finalize(prev) == int(warp)
        torch.cuda.synchronize(self.dev)
        u = lambda x: x.cpu().numpy().view(np.uint32)
        return rc, {"header": u(hdr), "tid": u(tid), "species": u(sp), "col_off": u(col), "first": u(first), "db_start": dbs.cpu().numpy().view(np.uint64),
                    "chunks": u(chunks).reshape(-1, 8), "max_chunks": max_chunks}

    def __call__(self, **kw):
        rc, got = self.call(**kw)
        native.check(rc)
        return got

    def ticket(self):
        """The "CTAs done" ticket behind the per-locus results in the scratch (u64 res_key[n_loci] | u32 res_first[n_loci] | pad to 8 | u32)."""
        off = (self.tb.n_loci * 12 + 7) & ~7
        return int(self.scratch[off:off + 4].cpu().numpy().view(np.uint32)[0])

    def tables(self):
        return (self.sum_as.cpu().numpy(), self.n_hit.cpu().numpy().view(np.uint32), self.first_idx.cpu().numpy().view(np.uint32),
                self.counters.cpu().numpy().view(np.uint64))


def assert_outputs(got, want, want_first=True, counters=None):
    """Every output word against the reference; the words past the outputs keep the driver's sentinel."""
    n, h = want["n"], got["header"]
    assert h[:5].tolist() == want["header"], (h[:5].tolist(), want["header"])
    assert h[5] == SENT and (h[10:] == SENT).all()
    if counters is None:
        assert (h[6:10] == SENT).all()
    else:
        assert int(h[6]) | int(h[7]) << 32 == counters[0] and int(h[8]) | int(h[9]) << 32 == counters[1]
    assert got["tid"][:n].tolist() == want["tid"] and (got["tid"][n:] == SENT).all()
    assert got["species"][:n].tolist() == want["species"] and (got["species"][n:] == SENT).all()
    if want_first:
        assert got["first"][:n].tolist() == want["first"]
    assert (got["first"][n if want_first else 0:] == SENT).all()
    assert got["col_off"][:n + 1].tolist() == want["col_off"] and (got["col_off"][n + 1:] == SENT).all()
    assert got["db_start"][:n].tolist() == want["db_start"] and (got["db_start"][n:] == (SENT | SENT << 32)).all()
    k = want["header"][1]
    assert [tuple(r) for r in got["chunks"][:k].tolist()] == want["chunks"]
    assert (got["chunks"][k:] == SENT).all()


# ------------------------------------------------------------------------------------------------ register window and remainder
def window_case(seed):
    """Ten loci in three species.  Loci of 1023, 1024, 1025, 2048, 2049 and 5000 rows with a unique winner at the given row of the locus
    (the last of the window, the first and last remainder rows, a row of the third remainder sweep); two loci of 1500 rows with an exact
    rounded tie between a window row and a remainder row, the lower allele number on the window side in one and on the remainder side in the
    other; a locus of 1100 rows whose maximum hit count only a remainder row holds (the penalty then applies to every window row, and the
    best unpenalized average sits in the window); one locus of 3 rows.  Allele numbers are shuffled against row order.
    -> Tables (rows grouped by locus), {locus: expected winner's index in the locus}."""
    rng = np.random.default_rng(seed)
    spec = [(1023, 1022), (1024, 1023), (1025, 1024), (2048, 2047), (2049, 2048), (5000, 3333), (1500, "tie_w"), (1500, "tie_r"),
            (1100, "max_r"), (3, 2)]
    locus_of, allele, s, n, expect = [], [], [], [], {}
    for l, (R, what) in enumerate(spec):
        a = rng.choice(np.arange(1, 4 * R + 1), R, replace=False).astype(np.int64)   # shuffled, not 1..R
        nn = np.where(rng.random(R) < 0.4, rng.integers(1, 61, R), 0).astype(np.int64)
        ss = nn * rng.integers(100, 140, R) + rng.integers(0, 5, R) * (nn > 0)
        nn[min(5, R - 2)], ss[min(5, R - 2)] = 80, 80 * 120   # the locus maximum hit count, in the window
        if isinstance(what, int):
            nn[what], ss[what] = 80, 80 * 150
            expect[l] = what
        elif what in ("tie_w", "tie_r"):
            w, r = 100, 1300                               # 150.0 and 150.0125: both round to 150.0
            nn[w], ss[w], nn[r], ss[r] = 80, 12000, 80, 12001
            lo, hi = sorted((a[w], a[r]))
            a[w], a[r] = (lo, hi) if what == "tie_w" else (hi, lo)
            expect[l] = w if what == "tie_w" else r
        else:                                              # max_r
            nn[5], ss[5] = 50, 50 * 200                    # 200 unpenalized; (10000 - 50 * 100) / 50 = 100 with the true maximum
            nn[nn > 60] = 60
            nn[1050], ss[1050] = 100, 100 * 150
            expect[l] = 1050
        locus_of += [l] * R
        allele.append(a)
        n.append(nn)
        s.append(ss)
    n, s = np.concatenate(n), np.concatenate(s)
    tb = Tables(locus_of, np.concatenate(allele), [0, 0, 0, 0, 1, 1, 1, 1, 2, 2], [4, 4, 2], s, n, unique_firsts(rng, n),
                counters=(1 << 40 | 5, 1 << 33 | 7), seed=seed)
    return tb, expect


@gpu
@pytest.mark.parametrize("interleaved", [False, True])
def test_register_window_and_remainder_rows(interleaved):
    rng = np.random.default_rng(11)
    tb, expect = window_case(11)
    if interleaved:
        tb = tb.interleaved(rng)
    assert tb.grouped != interleaved
    want = select_reference(tb)
    pos = tb.pos_in_locus()
    sizes = np.bincount(tb.locus_of.astype(np.int64))
    assert sorted(set(sizes.tolist()) & {1023, 1024, 1025, 2048, 2049, 5000}) == [1023, 1024, 1025, 2048, 2049, 5000]
    # the reference picks the constructed winners; which of them lie beyond the register window
    assert {l: int(pos[t]) for l, t in want["chosen_locus"].items()} == expect
    assert sum(1 for l, p in expect.items() if p >= WINDOW) == 6
    far_max = 8   # the max_r locus: its maximum hit count only beyond the window
    rows8 = np.nonzero(tb.locus_of == far_max)[0]
    mx = int(tb.n_hit[rows8].max())
    assert (pos[rows8[tb.n_hit[rows8] == mx]] >= WINDOW).all()
    assert want["n"] == 10 and not warp_finalizer(10, 3, 0) and warp_finalizer(10, 3, 1)
    sel = Selector(tb)
    for warp in (0, 1):
        assert_outputs(sel(warp=warp), want, counters=tb.counters)


# ------------------------------------------------------------------------------------------------ many loci and species
def random_index(seed, n_loci, n_species, max_alleles=6, interleave=False):
    """n_loci loci over n_species species (1 to 10 loci each where the shape allows it), 1 to max_alleles rows per locus, about 10 % of the
    loci without hits and some species with more `genes` rows than loci (they fail a strict gate)."""
    rng = np.random.default_rng(seed)
    sol = np.empty(n_loci, np.int64)
    k = min(n_loci, n_species)
    sol[:k] = rng.permutation(n_species)[:k]
    if n_loci > k:
        cap = max(10, -(-n_loci // n_species))
        cnt = np.bincount(sol[:k], minlength=n_species)
        for i in range(k, n_loci):   # at most `cap` loci per species
            while True:
                sp = int(rng.integers(0, n_species))
                if cnt[sp] < cap:
                    break
            sol[i] = sp
            cnt[sp] += 1
    sol = sol[rng.permutation(n_loci)]
    per = rng.integers(1, max_alleles + 1, n_loci)
    locus_of = np.repeat(np.arange(n_loci), per)
    nr = locus_of.shape[0]
    allele = np.empty(nr, np.int64)
    allele[:] = rng.integers(1, 1 << 31, nr)
    for l in np.nonzero(per > 1)[0]:   # unique inside a locus
        r0 = int(per[:l].sum())
        allele[r0:r0 + per[l]] = rng.choice(1 << 20, int(per[l]), replace=False) + 1
    nohit = rng.random(n_loci) < 0.1
    n = np.where((rng.random(nr) < 0.7) & ~nohit[locus_of], rng.integers(1, 200, nr), 0).astype(np.int64)
    s = np.where(n > 0, n * rng.integers(50, 200, nr) + rng.integers(-50, 50, nr), 0)
    loci_per_sp = np.bincount(sol, minlength=n_species)
    gdb = loci_per_sp + np.where(rng.random(n_species) < 0.3, rng.integers(1, 3, n_species), 0)
    gdb[gdb == 0] = 1
    tb = Tables(locus_of, allele, sol, gdb, s, n, unique_firsts(rng, n), counters=(int(rng.integers(0, 1 << 50)), 3), seed=seed)
    return tb.interleaved(rng) if interleave else tb


def largest_accepted(max_dynamic, n_species):
    return (max_dynamic - 16 - 4 * (1 + 4 * n_species)) // 44


@pytest.fixture(scope="module")
def max_dynamic():
    """The dynamic shared memory per block the library says the device allows, from its refusal of the largest declared shape."""
    tb = random_index(1, 4, 2)
    rc, _ = Selector(tb).call(n_loci=8192, n_species=4096)
    assert rc == native.E_RANGE
    msg = native.lib().mmlst_last_error().decode()
    m = re.fullmatch(r"mmlst_select_dev: 8192 loci / 4096 species need (\d+) bytes of shared memory per block for the selection, "
                     r"the device allows (\d+)", msg)
    assert m, msg
    need, allows = int(m.group(1)), int(m.group(2))
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    assert need == smem_bytes(8192, 4096) > optin and optin - 1024 <= allows < optin
    return allows


SHAPES = [(32, 32), (32, 1), (33, 1), (33, 33), (255, 32), (256, 33), (257, 200),
          ("fits 48 KB, not with the static part", 1), ("first past 48 KB", 1), ("first past 48 KB", 300), (3000, 400),
          ("largest", 700), ("largest", 4096)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "%s-%s" % s)
def test_many_loci_and_species(shape, max_dynamic):
    what, ns = shape
    if what == "fits 48 KB, not with the static part":   # the 128 bytes of static shared memory push the launch past the default limit
        nl = (DEFAULT_SMEM - 16 - 4 * (1 + 4 * ns)) // 44
        assert DEFAULT_SMEM - 128 < smem_bytes(nl, ns) <= DEFAULT_SMEM
    elif what == "first past 48 KB":
        nl = (DEFAULT_SMEM - 16 - 4 * (1 + 4 * ns)) // 44 + 1
        assert smem_bytes(nl, ns) > DEFAULT_SMEM >= smem_bytes(nl - 1, ns)
    elif what == "largest":
        nl = largest_accepted(max_dynamic, ns)
        assert smem_bytes(nl, ns) <= max_dynamic < smem_bytes(nl + 1, ns)
    else:
        nl = what
    tb = random_index(1000 + nl + ns, nl, ns, interleave=(nl + ns) % 2 == 1)
    if what in ("first past 48 KB", "largest") or nl >= 3000:   # the launches that must opt in to more than 48 KB
        assert smem_bytes(nl, ns) > DEFAULT_SMEM
    sel = Selector(tb)
    failed = 0
    for nloci in (100, 60):
        want = select_reference(tb, nloci=nloci)
        failed += len({int(tb.sol[l]) for l in want["chosen_locus"]}) - len(set(want["species"]))   # detected species that fail the gate
        assert len(want["chosen_locus"]) < nl                                                         # loci without hits
        assert want["n"] > 0 or nloci == 100
        for warp in ((0, 1) if nl <= 32 and ns <= 32 else (0,)):
            assert warp_finalizer(nl, ns, warp) == (warp == 1)
            assert_outputs(sel(nloci=nloci, warp=warp), want, counters=tb.counters)
    assert failed > 0
    if what == "largest":   # one more locus is refused before any launch, and the library goes on working
        rc, got = sel.call(n_loci=nl + 1)
        assert rc == native.E_RANGE and (got["header"] == SENT).all()
        assert native.lib().mmlst_last_error().decode() == (
            "mmlst_select_dev: %d loci / %d species need %d bytes of shared memory per block for the selection, the device allows %d"
            % (nl + 1, ns, smem_bytes(nl + 1, ns), max_dynamic))
        assert_outputs(sel(), select_reference(tb), counters=tb.counters)


def upload_index(ctx, nl, ns):
    lib = native.lib()
    locus_of = np.arange(nl, dtype=np.uint32)
    allele = np.ones(nl, np.uint32)
    sol = (np.arange(nl) % ns).astype(np.uint32)
    gdb = np.ones(ns, np.uint32)
    db_ascii = np.full(nl * 4 + 8, ord("A"), np.uint8)
    db_off = (np.arange(nl + 1) * 4).astype(np.uint64)
    ln = np.full(nl, 4, np.uint32)
    ix = native.Index(native.ptr(locus_of), native.ptr(allele), nl, native.ptr(sol), nl, native.ptr(gdb), ns, native.ptr(db_ascii),
                      native.ptr(db_off), native.ptr(ln))
    return lib.mmlst_index_upload(ctx.handle, C.byref(ix))


@gpu
def test_index_upload_refuses_what_the_selection_cannot_serve(max_dynamic):
    """mmlst_index_upload applies the selection's shared-memory bound: MMLST_E_RANGE with both sizes, not a CUDA error at the first sample."""
    ctx = native.Context(0)
    try:
        for nl, ns in ((8192, 4096), (largest_accepted(max_dynamic, 700) + 1, 700), (largest_accepted(max_dynamic, 4096) + 1, 4096)):
            assert upload_index(ctx, nl, ns) == native.E_RANGE
            assert native.lib().mmlst_last_error().decode() == (
                "mmlst_index_upload: %d loci / %d species need %d bytes of shared memory per block for the selection, the device allows %d"
                % (nl, ns, smem_bytes(nl, ns), max_dynamic))
        assert upload_index(ctx, largest_accepted(max_dynamic, 700), 700) == 0
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------------------ rounding at scale
def tie_candidates():
    """(final score F, hit count n, kind) with F / n on a tenths tie x.x5.  "exact": F / n is a binary tie (only x.25 / x.75 can be: n = 4,
    20, 2^k).  "near": F / n is a non-binary tie or one unit of F off it (n = 20 m, up to 2^32 - 1, |F| up to about 2^50), so the double
    quotient lies within one ulp of the tie (or within 2 / n) and Python's rounding follows the side it fell on.  Both signs."""
    out = []
    for n in (4, 20, 1 << 3, 1 << 10, 1 << 20, 1 << 31):
        for x in (Fraction(54101, 4), Fraction(3, 4), Fraction(-54101, 4), Fraction(-1, 4), Fraction(2 ** 32 + 1, 4)):
            F = x * n
            if F.denominator == 1 and abs(F) < 2 ** 51:
                out.append((int(F), n, "exact"))
    for n in (20, 20 * 123457, 4294967260, 0xFFFFFFFF):
        for T in (1351, -1351, 2_500_001, 1_000_003, -2_000_007):   # ties at T / 10 + 0.05
            for d in ((-1, 0, 1) if n > 20 else (0,)):
                F = n * (2 * T + 1) // 20 + d
                if abs(F) < 2 ** 51:
                    out.append((F, n, "near"))
    return out


def rounding_case(penalty):
    """Per candidate (allele 1) two loci, each with a rival (allele 2) whose average is exactly a tenth: one tenth above the candidate's
    rounded average (the rival wins; a candidate rounded one tenth up would tie and win on its allele number), and equal to it (the candidate
    wins the tie; rounded one tenth down it would lose).  The rival has 10 hits or the next multiple of 10 above the candidate's count, so
    the penalty falls on either side.  -> Tables, winner's row inside every locus (0 = candidate, 1 = rival)."""
    locus_of, allele, s, n, expect = [], [], [], [], []
    for i, (F, nA, _kind) in enumerate(tie_candidates()):
        T = int(round(Fraction(round(float(F) / float(nA), 1)) * 10))   # the candidate's rounded average, in tenths
        for dT in (1, 0):
            l = len(expect)
            up = (nA // 10 + 1) * 10
            nB = up if (i + dT) % 2 and up <= 0xFFFFFFFF else 10
            mx = max(nA, nB)
            locus_of += [l, l]
            allele += [1, 2]
            s += [F + (mx - nA) * penalty, (T + dT) * (nB // 10) + (mx - nB) * penalty]
            n += [nA, nB]
            expect.append(dT)
    nl = len(expect)
    n = np.asarray(n, np.int64)
    tb = Tables(locus_of, allele, np.zeros(nl, np.int64), [nl], s, n, unique_firsts(np.random.default_rng(penalty), n), seed=penalty)
    return tb, expect


def test_rounding_candidates_sit_on_tenths_ties():
    """Host check of the crafted values: the exact ones are binary ties, the near ones are not but lie within 2 / n of a tie (many within one
    ulp), and the counts and sums reach the extremes the kernel must handle."""
    c = tie_candidates()
    within_ulp = 0
    for F, n, kind in c:
        q = float(F) / float(n)
        t = Fraction(math.floor(Fraction(q) * 10) * 2 + 1, 20)   # the tie x.x5 next to q
        ulps = abs(Fraction(q) - t) / Fraction(math.ulp(q))
        if kind == "exact":
            assert ulps == 0 and Fraction(F, n) == t
        else:
            assert 0 < abs(Fraction(q) - t) <= Fraction(2, n) + Fraction(math.ulp(q))
            within_ulp += ulps <= 1
    assert within_ulp >= 15
    assert max(abs(F) for F, *_x in c) > 2 ** 49 and max(n for _F, n, _k in c) == 0xFFFFFFFF and min(F for F, *_x in c) < 0
    for penalty in (0, 1, 100, 10 ** 6):
        tb, expect = rounding_case(penalty)
        assert int(np.abs(tb.sum_as).max()) < 2 ** 62 and (tb.n_hit > 0).all() and set(expect) == {0, 1}
        penalized = tb.n_hit[0::2] < np.maximum(tb.n_hit[0::2], tb.n_hit[1::2])
        assert penalized.any() and not penalized.all()   # the candidate carries the penalty in some loci, the rival in others


@gpu
@pytest.mark.parametrize("penalty", [0, 1, 100, 10 ** 6])
def test_rounding_at_scale(penalty):
    tb, expect = rounding_case(penalty)
    want = select_reference(tb, penalty=penalty, nloci=0)
    pos = tb.pos_in_locus()
    assert [int(pos[want["chosen_locus"][l]]) for l in range(tb.n_loci)] == expect   # the rival wins exactly where it was built to
    assert int(tb.n_hit.max()) == 0xFFFFFFFF and int(np.abs(tb.sum_as).max()) > 2 ** 49
    assert_outputs(Selector(tb)(penalty=penalty, nloci=0), want, counters=tb.counters)


# ------------------------------------------------------------------------------------------------ gate
def gate_pairs():
    return [(d, t) for t in range(1, 101) for d in range(1, t + 1)]


def gate_case(pairs, seed):
    """One species per (detected, genes) pair: `detected` loci of one hit row each, plus one locus without hits when detected < genes."""
    rng = np.random.default_rng(seed)
    sol, hit = [], []
    for sp, (d, t) in enumerate(pairs):
        sol += [sp] * d
        hit += [True] * d
        if d < t:
            sol.append(sp)
            hit.append(False)
    nl = len(sol)
    n = np.asarray(hit, np.int64)
    return Tables(np.arange(nl), np.ones(nl, np.int64), sol, [t for _d, t in pairs], n * 100, n, unique_firsts(rng, n), seed=seed)


def gate_threshold(d, t):
    return int((float(d) / float(t)) * 100)


def test_gate_thresholds_cover_float_artifacts():
    """Host check: the (detected, genes) pairs include thresholds where (d / t) * 100 falls just under an integer, e.g. 29 / 100."""
    odd = [(d, t) for d, t in gate_pairs() if gate_threshold(d, t) != d * 100 // t]
    assert (29, 100) in odd and len(odd) >= 4
    assert gate_threshold(29, 100) == 28


@gpu
def test_gate_at_every_detected_count():
    """genes_in_db 1-100, every detected count 1..genes, nloci at, one below and one above the threshold int((d / t) * 100): every species is
    run at the three values (grouped by nloci so that one call checks many species)."""
    by_x = {}
    for d, t in gate_pairs():
        v = gate_threshold(d, t)
        for x in (v - 1, v, v + 1):
            by_x.setdefault(x, []).append((d, t))
    checked = 0
    for x, pairs in sorted(by_x.items()):
        batch, loci = [], 0
        for p in pairs + [None]:
            if p is not None and loci + p[0] + 1 <= 3000:
                batch.append(p)
                loci += p[0] + 1
                continue
            tb = gate_case(batch, x)
            want = select_reference(tb, nloci=x)
            kept = set(want["species"])
            assert kept == {sp for sp, (d, t) in enumerate(batch) if gate_threshold(d, t) >= x}
            assert_outputs(Selector(tb)(nloci=x), want, counters=tb.counters)
            checked += len(batch)
            batch, loci = ([p], p[0] + 1) if p is not None else ([], 0)
    assert checked == 3 * len(gate_pairs())


@gpu
def test_gate_broken_database_and_local_flag():
    """tot < det sets error bit 1 and drops that species only; MMLST_SELECT_LOCAL disables the gate (and the check)."""
    tb = gate_case([(3, 3), (2, 4), (4, 3), (1, 1), (2, 1), (5, 10)], 5)
    for warp in (0, 1):
        sel = Selector(tb)
        for nloci, flags in ((100, 0), (50, 0), (0, 0), (100, LOCAL), (50, LOCAL)):
            want = select_reference(tb, nloci=nloci, flags=flags)
            assert want["header"][3] == (0 if flags else 1)
            assert set(want["species"]) == ({0, 1, 2, 3, 4, 5} if flags else {0, 3} | ({1, 5} if nloci <= 50 else set()))
            assert_outputs(sel(nloci=nloci, flags=flags, warp=warp), want, counters=tb.counters)


# ------------------------------------------------------------------------------------------------ outputs
@gpu
@pytest.mark.parametrize("shape", [(30, 9), (300, 70)])
@pytest.mark.parametrize("chunk_records", [512, 1536, 0])
def test_outputs_chunk_list_and_overflow(shape, chunk_records):
    """Header, chosen rows / species / first records, columns, DB offsets and the chunk list, with pileup record counts from 0 to 20 000 per
    row (0 = one empty chunk for a chosen locus), at max_chunks = the need (bit 2 clear) and one below (bit 2 set, header[1] = max_chunks,
    the listed chunks still right); without chosen_first or counters those outputs stay untouched."""
    nl, ns = shape
    tb = random_index(77 + nl, nl, ns)
    rng = np.random.default_rng(nl)
    tb.nrec = np.where(rng.random(tb.n_ref) < 0.15, 0, rng.integers(1, 20000, tb.n_ref)).astype(np.int64)
    sel = Selector(tb)
    want = select_reference(tb, nloci=50, chunk_records=chunk_records)
    need = want["n_chunks_needed"]
    chosen_nrec = [int(tb.nrec[t]) for t in want["tid"]]
    assert 0 in chosen_nrec and max(chosen_nrec) > 3 * want["header"][4]   # an empty chunk, and loci of several chunks
    if chunk_records == 0:
        assert want["header"][4] == native.lib().mmlst_chunk_records(sum(chosen_nrec))
    for warp in ((0, 1) if nl <= 32 else (0,)):
        for mc in (need, need - 1):
            w = select_reference(tb, nloci=50, chunk_records=chunk_records, max_chunks=mc)
            assert (w["header"][3] & 2) == (2 if mc < need else 0) and w["header"][1] == mc
            assert_outputs(sel(nloci=50, chunk_records=chunk_records, max_chunks=mc, warp=warp), w, counters=tb.counters)
        assert_outputs(sel(nloci=50, chunk_records=chunk_records, max_chunks=need, warp=warp, want_first=False, want_counters=False),
                       select_reference(tb, nloci=50, chunk_records=chunk_records, max_chunks=need), want_first=False)


# ------------------------------------------------------------------------------------------------ consume and reuse
@gpu
@pytest.mark.parametrize("warp", [0, 1])
@pytest.mark.parametrize("interleaved", [False, True])
def test_consume_resets_every_row_and_the_next_call_is_clean(warp, interleaved):
    """MMLST_SELECT_CONSUME leaves every row of every locus (remainder rows too) at sum 0, hits 0, first index 0xFFFFFFFF, the counters at 0
    and the scratch's CTA ticket at zero; a second call on new tables with MMLST_SELECT_SCRATCH_CLEAN (no ticket memset) gives the reference's answer:
    what a cohort of samples typed back to back relies on."""
    tb, _ = window_case(3)
    nxt, _ = window_case(4)   # same loci sizes: new score tables for the same rows
    nxt = tb.with_scores(nxt.sum_as, nxt.n_hit, nxt.first_idx, (123, 45))
    if interleaved:
        tb, nxt = tb.interleaved(np.random.default_rng(5)), nxt.interleaved(np.random.default_rng(5))
        assert np.array_equal(tb.locus_of, nxt.locus_of) and np.array_equal(tb.allele_num, nxt.allele_num)
    assert ((tb.n_hit > 0) & (tb.pos_in_locus() >= WINDOW)).sum() > 1000   # hit rows the remainder loops reset
    sel = Selector(tb)
    flags = CONSUME | SCRATCH_CLEAN
    assert_outputs(sel(flags=flags, warp=warp), select_reference(tb), counters=tb.counters)
    s, n, f, c = sel.tables()
    assert not s.any() and not n.any() and (f == NO_IDX).all() and not c.any()
    assert sel.ticket() == 0
    sel.load(nxt)
    assert_outputs(sel(flags=flags, warp=warp), select_reference(nxt), counters=nxt.counters)
    s, n, f, c = sel.tables()
    assert not s.any() and not n.any() and (f == NO_IDX).all() and not c.any()


# ------------------------------------------------------------------------------------------------ end to end
def db_shape_case():
    """34 species of 1 to 7 loci, 3 alleles per locus except two loci of 1100 and 1030 alleles whose strain allele (where the reads land)
    is row 1076 / 1029 of the locus; two species list one more gene than they have loci (they fail the 100 % gate)."""
    from metamlst_b200 import synth
    rng = np.random.default_rng(2024)
    orgs = ["sp%02d" % i for i in range(34)]
    schemes = {o: [("g%d" % j, int(rng.integers(300, 420))) for j in range(1 + i % 7)] for i, o in enumerate(orgs)}
    big = {("sp00", "g0"): (1100, 1077), ("sp05", "g3"): (1030, 1030)}   # (alleles, allele variant of the sample's strain)
    apl = [big.get((o, g), (3, 0))[0] for o in orgs for g, _ln in schemes[o]]
    db = synth.make_db(orgs, alleles_per_locus=apl, n_profiles=4, seed=2024, schemes=schemes)
    for (o, g), (_n, v) in big.items():
        db.profiles[o][:, [g for g, _ln in schemes[o]].index(g)] = v
    gdb = {o: len(schemes[o]) + (1 if i in (9, 20) else 0) for i, o in enumerate(orgs)}
    return db, gdb, big


def tables_of(index, gdb, ref_lens, tables):
    """Tables of a finished pass (sum_as, n_hit, first_idx) over the pass's index, species in order of first locus (as the library numbers them)."""
    names = list(dict.fromkeys(sp for sp, _g in index.locus_names))
    sol = [names.index(sp) for sp, _g in index.locus_names]
    s, n, f = tables
    return names, Tables(index.locus_of, [int(a) for a in index.allele], sol, [gdb[sp] for sp in names], s, n, f, ref_len=ref_lens)


@gpu
def test_database_shape_end_to_end():
    """DevicePipeline (eager and captured graph, score tables kept) and the one-call path (mmlst_sample through api.type_soa) on a DB of more
    than 32 species whose reads land on allele rows beyond the register window: chosen contigs and their order equal the reference applied
    to the pass's own score tables, and every consensus equals the C port's (`corc.consensus` over `corc.contig_counts`)."""
    from metamlst_b200 import devpack, pipeline, synth
    from oracle import corc
    db, gdb, big = db_shape_case()
    index = api.AlleleIndex(db.ref_names())
    assert len(db.organisms) > 32 and index.n_loci <= 8 * 34
    big_rows = {}
    for (o, g), (n_all, v) in big.items():
        li = db.locus_names.index((o, g))
        assert int(db.locus_row0[li + 1] - db.locus_row0[li]) == n_all > WINDOW and v - 1 >= WINDOW
        big_rows[li] = int(db.locus_row0[li])
    n_reads, gk = 30000, dict(read_len=100, seed=91, K=4, sub_err=0.01, novel_loci=0)
    st = devpack.pack_cores(db, [synth.gen_core(db, n_reads, device="cuda:0", **gk)], 20, 8000)
    stab = synth.make_sample(db, n_reads, device="cuda:0", **gk).sorted_by_coord()
    kw = dict(minscore=170, max_xM=4, nloci=100)

    def expected(tables):
        names, tb = tables_of(index, gdb, st.ref_lens, tables)
        want = select_reference(tb)
        for li, r0 in big_rows.items():   # the winners of the big loci lie beyond the register window
            assert want["chosen_locus"][li] - r0 >= WINDOW
        assert len(set(want["species"])) < len(db.organisms) and len(set(want["species"])) > 32 - 2
        out = []
        for sp, t in zip(want["species"], want["tid"]):
            if not out or out[-1][0] != names[sp]:
                out.append((names[sp], []))
            out[-1][1].append(index.ref_names[t])
        return out

    def check_consensus(species):
        for _sp, lst in species:
            for contig, seq, holes, snps in lst:
                t = index.name_to_tid[contig]
                counts, _ = corc.contig_counts(stab, t, 20, kw["minscore"], kw["max_xM"], 8000)
                assert (seq, holes, snps) == corc.consensus(counts, db.row_seq(t).encode(), 1)

    pipe = pipeline.DevicePipeline(st, index, db.row_seq, genes_in_db=gdb, **kw)
    pipe.want_tables = True
    a = pipe.step()
    got = [(sp, [c for c, *_x in lst]) for sp, lst in a.items()]
    assert got == expected(pipe.tables())
    check_consensus(a.items())
    pipe.capture()
    assert pipe.step_graph() == a and expected(pipe.tables()) == got
    ctx = native.Context(0)
    try:
        sidx = api.SampleIndex(ctx, index, st.ref_lens, db.row_seq, genes_in_db=gdb)
        r = api.type_soa(sidx, st.to_host(pinned=True), min_read_len=50, penalty=100, want_tables=True, **kw)
        assert [(sp, [c for c, *_x in lst]) for sp, lst in r["species"]] == expected(r["tables"]) == got
        assert r["species"] == list(a.items())
    finally:
        ctx.close()
