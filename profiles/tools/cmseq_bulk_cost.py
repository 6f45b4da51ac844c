"""Cost of cmseq's whole-BAM statistics (cmseq_api.BamFile *_all methods) against the per-contig loop, and of the contig-statistics kernels
(csrc/contig_stats.cu) against their algorithmic bytes over the measured HBM copy rate.

    python profiles/tools/cmseq_bulk_cost.py --out profiles/cmseq_bulk_cost.json [--contigs 3000] [--reps 3]

On the seeded many-contig BAM of tests/test_cmseq_bulk.py (write_many_contig_bam), for each of the four statistics: the wall time of
`{name: contig.method(...) for every contig}` and of the bulk method (median of --reps, after one warm-up of each), and the equality of
the two results.  Kernel: mmlst_contig_stats_dev over a device count tensor of --kernel-cols random columns (larger than the L2), CUDA
events around 20 calls per mode.  The card's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def hbm_copy_rate(torch, nbytes=4 << 30):
    a = torch.empty(nbytes // 4, dtype=torch.int32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * 10 / (e0.elapsed_time(e1) * 1e-3)   # read + write


def kernel_cost(torch, native, total, copy_rate):
    lib = native.lib()
    rng = np.random.default_rng(1)
    lens = rng.integers(1, 4000, total // 2000 + 10)
    col_off = np.zeros(lens.size + 1, np.int64)
    col_off[1:] = np.cumsum(lens)
    n = int(np.searchsorted(col_off, total, side="right") - 1)
    col_off = col_off[:n + 1].astype(np.uint32)
    total = int(col_off[-1])
    dev = "cuda"
    counts = torch.randint(0, 8, (total, 5), dtype=torch.int32, device=dev)
    counts[torch.randint(0, total, (total // 4,), device=dev)] = 0   # a quarter of the columns uncovered
    d_off = torch.from_numpy(col_off.view(np.int32)).to(dev)
    scratch = torch.empty(int(lib.mmlst_contig_stats_scratch_bytes(total)), dtype=torch.uint8, device=dev)
    sel, low = torch.empty(n + 1, dtype=torch.int32, device=dev), torch.empty(n + 1, dtype=torch.int32, device=dev)
    dep = torch.empty(n + 1, dtype=torch.int64, device=dev)
    oc = torch.empty(total, dtype=torch.int32, device=dev)
    ov = torch.empty(total * 5, dtype=torch.int32, device=dev)
    cons = torch.empty(total, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    for mode, name, width, want_cons in ((native.STATS_COLUMNS, "columns", 5, False), (native.STATS_DEPTH, "depth", 1, False),
                                         (native.STATS_LOWDOM, "lowdom+consensus", 2, True)):
        prm = native.ContigStatsParams(mode, 2, 0, ord("-"), 0.8)

        def call():
            native.check(lib.mmlst_contig_stats_dev(native.ptr(counts), native.ptr(d_off), n, total, C.byref(prm), native.ptr(scratch),
                                                    scratch.numel(), native.ptr(sel), native.ptr(low), native.ptr(dep), native.ptr(oc),
                                                    native.ptr(ov), native.ptr(cons) if want_cons else None, 0, st))
        call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            call()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3 / 20
        k = int((low if mode == native.STATS_LOWDOM else sel)[-1].item())
        algo = 20 * total + (total if want_cons else 0) + 4 * (1 + width) * k + 16 * (n + 1)
        out[name] = {"columns": total, "contigs": n, "compacted": k, "kernel_s": t, "algorithmic_bytes": algo,
                     "floor_s_at_copy_rate": algo / copy_rate, "share_of_copy_rate": algo / copy_rate / t}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--contigs", type=int, default=3000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-cols", type=int, default=100_000_000)
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from metamlst_b200 import cmseq_api, native
    from test_cmseq_bulk import _same, write_many_contig_bam

    res = {"card": card()}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "many.bam")
        write_many_contig_bam(path, n_contigs=a.contigs)
        bf = cmseq_api.BamFile(path)
        res["contigs"] = len(bf.contigs)
        res["columns"] = int(sum(c.length for c in bf.contigs.values()))
        tagf = [("AS", "loc_gte", 80), ("XM", "loc_lte", 5)]
        stats = {"get_base_stats": ("base_stats_all", {"min_read_depth": 1, "BAM_tagFilter": tagf}),
                 "reference_free_consensus": ("reference_free_consensus_all", {"mincov": 1}),
                 "polymorphism_rate": ("polymorphism_rate_all", {"mincov": 2}),
                 "breadth_and_depth_of_coverage": ("breadth_and_depth_of_coverage_all", {"mincov": 1, "trunc": 10})}
        res["statistics"] = {}
        for method, (bulk, kw) in stats.items():
            loop = lambda: {n: getattr(c, method)(**kw) for n, c in bf.contigs.items()}
            whole = lambda: getattr(bf, bulk)(**kw)
            want, got = loop(), whole()   # warm-up; also the equality at the timed size
            _same(got, want)
            tl, tb = [], []
            for _ in range(a.reps):
                t0 = time.perf_counter(); loop(); tl.append(time.perf_counter() - t0)
                t0 = time.perf_counter(); whole(); tb.append(time.perf_counter() - t0)
            res["statistics"][method] = {"kwargs": {k: v for k, v in kw.items()}, "per_contig_loop_s": float(np.median(tl)),
                                         "bulk_s": float(np.median(tb)), "speedup": float(np.median(tl) / np.median(tb)), "outputs_equal": True}
            print(method, res["statistics"][method], flush=True)
        bf.close()
    rate = hbm_copy_rate(torch)
    res["hbm_copy_rate_Bps"] = rate
    res["kernel"] = kernel_cost(torch, native, a.kernel_cols, rate)
    res["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["kernel"], indent=1))
    print("card:", res["card"])


if __name__ == "__main__":
    main()
