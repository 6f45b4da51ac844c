"""Form 7 of the score kernel (the compact 2 B / record stream) against form 6 (3 B / record) on the bench's workload: two configs[1]
samples of bench.py's generator (40 M records each; launches alternate between them, so every launch streams from HBM), the kernel
time of each form over rounds that alternate the two forms, the algorithmic bytes and rate of each form against the device copy rate
measured here, the cost of deriving the compact stream (mmlst_score_pack16_dev) per sample and the HBM it adds, and the chunks form 7
reduces from the 3-byte arrays (per-chunk fallback) on the bench samples and on every golden BAM.  Card name and power limit are read
in the same run.

    python profiles/tools/score_compact_cost.py --out profiles/score_compact_cost.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))

from ingest_crc_cost import card, copy_rate  # noqa: E402


def events_ms(torch, fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
    cli = ap.parse_args()
    import numpy as np
    import torch
    sys.argv = ["bench.py"]
    import bench
    from metamlst_b200 import api, bam, native, pipeline
    args = bench.parse()
    lib = native.lib()
    dev = "cuda:0"
    out = {"card": card(), "copy_rate_GBps": copy_rate(torch) / 1e9}
    db = bench.make_db(args)
    index = api.AlleleIndex(db.ref_names())
    sts = [bench.gen_streams(db, args, dev, args.max_depth or None, None, seed=s)[0] for s in (1002, 1102)]
    pipes = [pipeline.DevicePipeline(st, index, db.row_seq, **bench.PARAMS) for st in sts]
    n = int(sts[0].as0.shape[0])
    n_runs, n_chunks = int(sts[0].run_tid.shape[0]), int(sts[0].chunk_run.shape[0])
    out["records"], out["runs"], out["chunks"] = n, n_runs, n_chunks
    out["fallback_chunks_bench"] = [p.compact_fallback_chunks() for p in pipes]

    # deriving the compact stream: what rebind() adds per sample (reads as0 + xm3 + chunk_qlen, writes code + head)
    for p in pipes:
        p._pack16()
    pack_ms = events_ms(torch, lambda i: pipes[i % 2]._pack16(), cli.reps)
    pack_bytes = 3.0 * n + 2.0 * n_chunks + 2.0 * n + 4.0 * n_chunks
    out["pack"] = {"ms": pack_ms, "bytes": pack_bytes, "GBps": pack_bytes / pack_ms / 1e6, "extra_hbm_bytes": 2.0 * 256 * ((n + 255) // 256) + 4.0 * ((n + 255) // 256)}

    # the two forms, alternating rounds; tables checked equal
    prev = lib.mmlst_set_score_variant(-1)
    times = {7: [], 6: []}
    tabs = {}
    for r in range(cli.rounds):
        for v in ((7, 6) if r % 2 == 0 else (6, 7)):
            lib.mmlst_set_score_variant(v)
            pipes[0].reset_tables()
            pipes[0]._score_call()
            torch.cuda.synchronize()
            tabs.setdefault(v, [pipes[0].zscore.clone(), pipes[0].first_idx.clone()])
            for p in pipes:
                p._score_call()
            times[v].append(events_ms(torch, lambda i: pipes[i % 2]._score_call(), cli.reps))
    lib.mmlst_set_score_variant(prev)
    assert all(torch.equal(a, b) for a, b in zip(tabs[7], tabs[6])), "form 7 and form 6 tables differ"
    alg = {7: 2.0 * n + 8.0 * n_runs + 8.0 * n_chunks, 6: 3.0 * n + 8.0 * n_runs + 6.0 * n_chunks}
    out["score"] = {}
    for v in (7, 6):
        ms = float(np.median(times[v]))
        out["score"]["form%d" % v] = {"ms_median": ms, "ms_all": times[v], "algorithmic_bytes": alg[v], "GBps": alg[v] / ms / 1e6,
                                     "frac_of_copy_rate": alg[v] / ms / 1e6 / out["copy_rate_GBps"]}
    out["score"]["ratio_form7_over_form6"] = out["score"]["form7"]["ms_median"] / out["score"]["form6"]["ms_median"]

    # golden BAMs: chunks form 7 would take from the 3-byte arrays at minscore 80 (-1: no compact stream, e.g. a file-order index)
    golden = os.path.join(ROOT, "tests", "golden")
    man = json.load(open(os.path.join(golden, "manifest.json")))
    gb = {}
    for name in sorted(man):
        path = os.path.join(golden, name, "sample.bam")
        if not os.path.exists(path):
            continue
        try:
            st = bam.ingest_bam(path, 0, presorted=man[name].get("order") == "coord")
        except native.MmlstError as e:
            gb[name] = {"refused": str(e)}
            continue
        gi = api.AlleleIndex(list(st.ref_names))
        p = pipeline.DevicePipeline(st, gi, lambda t: "A" * int(st.ref_lens[t]), **bench.PARAMS)
        gb[name] = {"records": int(st.as0.shape[0]), "full_chunks": int(st.as0.shape[0]) // 256, "fallback_chunks": p.compact_fallback_chunks()}
    out["fallback_chunks_golden"] = gb
    with open(cli.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "pack", "fallback_chunks_bench")}), json.dumps(out["score"]["ratio_form7_over_form6"]))


if __name__ == "__main__":
    main()
