"""Cost of cmseq's BamFile on the two ingest routes: ingest="host" (host unpacker, each batch uploaded) against ingest="device" (the
compressed file inflated and parsed on the GPU, the streams resident in HBM, mmlst_contig_stats_resident).

    python profiles/tools/cmseq_device_cost.py --out profiles/cmseq_device_cost.json [--contigs 100000] [--records 20000000] [--reps 1]

Two inputs: the seeded 3006-contig BAM of tests/test_cmseq_bulk.py (write_many_contig_bam) and a larger seeded coordinate-sorted BAM of
--contigs contigs and --records 50-base reads (written here with numpy, BGZF level 1).  For each route: the open time of
BamFile(path, ingest=...) -- disk read included; the file was just written, so it is read from the page cache -- and, for each of the four
statistics of cmseq_bulk_cost.py, the wall time of the whole-BAM method (median of --reps; on the 3006-contig BAM after one warm-up
call, which also warms every path for the large one).  The two routes' outputs are
asserted equal at the timed size.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import struct
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))

L = 50   # read length of the large input


def _bgzf(data) -> bytes:
    co = zlib.compressobj(1, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    return (struct.pack("<BBBBIBBHBBHH", 0x1F, 0x8B, 8, 4, 0, 0, 0xFF, 6, 66, 67, 2, len(comp) + 25) + comp +
            struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def write_large_bam(path, n_contigs, n_records, seed=7, chunk=1 << 20):
    """Coordinate-sorted BAM: contigs of 50..100 columns, reads of L bases copied from a random reference with 2 % substitutions, random
    qualities 2..40, aux AS:s XS:s XN:C XM:C (bowtie2's first four fields; AS = 100 - 6 XM, so the AS >= 80 / XM <= 5 filter keeps the reads
    with at most 3 substitutions).  Record layout fixed: 36 + 11 + 4 + L/2 + L + 18 bytes."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(L, 101, n_contigs)
    names = ["c%06d" % i for i in range(n_contigs)]
    ref = rng.integers(0, 4, int(lens.sum())).astype(np.uint8)
    ref_off = np.concatenate([[0], np.cumsum(lens)[:-1]])
    w = lens.astype(np.float64) - L + 1
    tid = np.sort(rng.choice(n_contigs, n_records, p=w / w.sum())).astype(np.int64)
    pos = (rng.random(n_records) * (lens[tid] - L + 1)).astype(np.int64)
    order = np.lexsort((pos, tid))
    tid, pos = tid[order], pos[order]
    text = ("@HD\tVN:1.0\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (n, l) for n, l in zip(names, lens))).encode()
    head = [b"BAM\1", struct.pack("<i", len(text)), text, struct.pack("<i", n_contigs)]
    for n, l in zip(names, lens):
        head.append(struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", int(l)))
    head = b"".join(head)
    rec = 36 + 11 + 4 + (L + 1) // 2 + L + 18
    per_block = 0xFF00 // rec
    code = np.array([1, 2, 4, 8], np.uint8)   # A C G T in BAM's 4-bit alphabet
    with open(path, "wb") as fh, ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        fh.write(b"".join(_bgzf(head[i:i + 0xFF00]) for i in range(0, len(head), 0xFF00)))
        for c0 in range(0, n_records, chunk):
            t, p = tid[c0:c0 + chunk], pos[c0:c0 + chunk]
            m = t.size
            b = np.zeros((m, rec), np.uint8)

            def put(col, vals, nbytes):
                v = np.asarray(vals, dtype=np.int64)
                for i in range(nbytes):
                    b[:, col + i] = (v >> (8 * i)) & 0xFF
            put(0, np.full(m, rec - 4), 4); put(4, t, 4); put(8, p, 4)
            b[:, 12] = 11; b[:, 13] = 42
            put(14, 4681 + (p >> 14), 2); put(16, np.ones(m), 2); put(18, np.zeros(m), 2); put(20, np.full(m, L), 4)
            put(24, np.full(m, -1), 4); put(28, np.full(m, -1), 4)
            ids = np.arange(c0, c0 + m)
            b[:, 36] = ord("r")
            for d in range(9, 0, -1):
                b[:, 36 + d] = 48 + ids % 10
                ids = ids // 10
            put(47, np.full(m, L << 4), 4)
            bases = ref[(ref_off[t] + p)[:, None] + np.arange(L)[None, :]]
            mut = rng.random((m, L)) < 0.02
            bases[mut] = rng.integers(0, 4, int(mut.sum()))
            nib = code[bases]
            b[:, 51:51 + L // 2] = (nib[:, 0::2] << 4) | nib[:, 1::2]
            q0 = 51 + (L + 1) // 2
            b[:, q0:q0 + L] = rng.integers(2, 41, (m, L))
            a0 = q0 + L
            xm = mut.sum(axis=1)
            for tag, typ, val, nb in ((b"AS", b"s", 100 - 6 * xm, 2), (b"XS", b"s", 90 - 6 * xm, 2), (b"XN", b"C", np.zeros(m), 1),
                                     (b"XM", b"C", xm, 1)):
                b[:, a0] = tag[0]; b[:, a0 + 1] = tag[1]; b[:, a0 + 2] = typ[0]
                put(a0 + 3, val, nb)
                a0 += 3 + nb
            flat = b.reshape(-1)
            spans = [(i * rec, min(m, i + per_block) * rec) for i in range(0, m, per_block)]
            fh.write(b"".join(pool.map(lambda ab: _bgzf(flat[ab[0]:ab[1]].tobytes()), spans)))
        fh.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))


STATS = {"get_base_stats": ("base_stats_all", {"min_read_depth": 1, "BAM_tagFilter": [("AS", "loc_gte", 80), ("XM", "loc_lte", 5)]}),
         "reference_free_consensus": ("reference_free_consensus_all", {"mincov": 1}),
         "polymorphism_rate": ("polymorphism_rate_all", {"mincov": 2}),
         "breadth_and_depth_of_coverage": ("breadth_and_depth_of_coverage_all", {"mincov": 1, "trunc": 10})}


def measure(path, reps, warmup):
    import torch
    from metamlst_b200 import cmseq_api
    from test_cmseq_bulk import _same
    out = {"bam_bytes": os.path.getsize(path)}
    handles = {}
    for route in ("host", "device"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        handles[route] = cmseq_api.BamFile(path, ingest=route)
        torch.cuda.synchronize()
        out.setdefault("open_s", {})[route] = time.perf_counter() - t0
    h, d = handles["host"], handles["device"]
    assert list(h.contigs) == list(d.contigs)
    s = d._soas[cmseq_api.CMSEQ_DEFAULTS.minqual]
    out.update(contigs=len(h.contigs), columns=int(sum(c.length for c in h.contigs.values())), records=int(s.tid.shape[0]),
               pileup_records=int(s.n_prec))
    out["statistics"] = {}
    for method, (bulk, kw) in STATS.items():
        row = {"kwargs": kw}
        got = {}
        for r in ("host", "device"):
            if warmup:
                getattr(handles[r], bulk)(**kw)
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                got[r] = getattr(handles[r], bulk)(**kw)
                ts.append(time.perf_counter() - t0)
            row[r + "_s"] = float(np.median(ts))
        _same(got["device"], got["host"])   # the equality at the timed size
        row["outputs_equal"] = True
        del got
        out["statistics"][method] = row
        print(os.path.basename(path), method, row, flush=True)
    for b in handles.values():
        b.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--contigs", type=int, default=100_000)
    ap.add_argument("--records", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=1)
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from cmseq_bulk_cost import card
    from test_cmseq_bulk import write_many_contig_bam
    res = {"card": card(), "routes": {"host": "bam.unpack_bam + mmlst_contig_stats (upload per batch)",
                                     "device": "bam.ingest_bam(lenient_tags, check_crc) + mmlst_contig_stats_resident"},
           "multi_gpu": "not measured"}
    def save():
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(res, f, indent=1)
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "many.bam")
        write_many_contig_bam(p)
        res["many_contig_bam"] = measure(p, a.reps, warmup=True)   # also warms every path of both routes
        save()
        os.remove(p)
        p = os.path.join(td, "large.bam")
        t0 = time.perf_counter()
        write_large_bam(p, a.contigs, a.records)
        print("wrote", p, os.path.getsize(p), "bytes in", time.perf_counter() - t0, "s", flush=True)
        res["large_bam"] = measure(p, a.reps, warmup=False)
        res["large_bam"]["generator"] = {"contigs": a.contigs, "records": a.records, "read_length": L, "seed": 7}
    res["card_after"] = card()
    save()
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
