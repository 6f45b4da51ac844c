"""Added cost of the BGZF CRC-32 check of the device ingest (`bam.ingest_bam(check_crc=True)`, csrc/ingest.cu crc_kernel) on the
bench's ingest workload: the BAM of bench.py's `ingest` leg (same generator and seed, 2 M reads x K=4 = 8 M records), in bowtie2 (name)
order and coordinate order, from page-locked memory.  Calls with the check off and on alternate (the order flips every round), so
drift on a shared machine hits both alike.  Reported per order: host wall time around the synchronous call (min / median / spread),
the per-phase device times of the library (CUDA events; the kernel counts in `inflate`), the kernel's own time from a separate
torch.profiler pass, and that time against the HBM floor (inflated bytes / the copy rate measured here).  Card name and power limit
are read in the same run.

    python profiles/tools/ingest_crc_cost.py --out profiles/ingest_crc_cost.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=60).stdout.decode().strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%r)" % e}


def copy_rate(torch, nbytes=4 << 30, reps=10):
    """Device-to-device copy of nbytes: bytes read + written per second (the HBM rate a streaming kernel can reach)."""
    x = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
    y = torch.empty_like(x)
    y.copy_(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = None
    for _ in range(reps):
        e0.record()
        y.copy_(x)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    del x, y
    torch.cuda.empty_cache()
    return 2.0 * nbytes / (best * 1e-3)


def stats(xs):
    import numpy as np
    a = np.asarray(xs, dtype=np.float64)
    med = float(np.median(a))
    return {"min_ms": float(a.min()) * 1e3, "median_ms": med * 1e3, "max_ms": float(a.max()) * 1e3, "spread": float((a.max() - a.min()) / med), "n": int(a.size)}


def kernel_ms(torch, bam, pinned, calls=3):
    """Mean device time of crc_kernel over `calls` ingests, from a torch.profiler trace (a run of its own: tracing slows the host)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            st = bam.ingest_bam(pinned, 0, check_crc=True)
            del st
        torch.cuda.synchronize()
    ks = [k for k in prof.key_averages() if "crc_kernel" in k.key]
    if not ks:
        return None
    k = ks[0]
    total_us = getattr(k, "device_time_total", None)
    if total_us is None:
        total_us = k.cuda_time_total
    return total_us / k.count * 1e-3, int(k.count)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7, help="calls per setting and order (alternating)")
    ap.add_argument("--ingest-reads", type=int, default=2_000_000, help="reads of the BAM (x K=4 records), as bench.py --ingest-reads")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    import numpy as np
    import torch
    sys.argv = sys.argv[:1]
    import bench
    from metamlst_b200 import bam, synth
    assert torch.cuda.is_available(), "needs a CUDA device"
    args = bench.parse()
    torch.cuda.set_device(0)
    res = {"card": card(), "hbm_copy_rate_GBps": copy_rate(torch) / 1e9, "workload": "bench.py ingest leg: %d reads x K=%d, seed 1002, align_records" % (a.ingest_reads, args.k)}
    db = bench.make_db(args)
    for order in ("name", "coord"):
        cores = bench.gen_cores(db, args, "cuda:0", None, seed=1002, n_reads=a.ingest_reads)
        raw = synth.write_bam_fast(db, cores, order=order, align_records=True)
        del cores
        torch.cuda.empty_cache()
        pinned = torch.from_numpy(raw.copy()).pin_memory()
        for flag in (False, True):   # warm-up: driver entry points, workspace cache
            st = bam.ingest_bam(pinned, 0, check_crc=flag)
            del st
        torch.cuda.synchronize()
        wall = {False: [], True: []}
        phases = {False: [], True: []}
        ing = None
        for i in range(a.reps):
            for flag in ((False, True) if i % 2 == 0 else (True, False)):
                t0 = time.perf_counter()
                st = bam.ingest_bam(pinned, 0, check_crc=flag)
                torch.cuda.synchronize()
                wall[flag].append(time.perf_counter() - t0)
                phases[flag].append(st.ingest_seconds)
                ing, n_rec = st.ingest_stats, int(st.tid.shape[0])
                del st
        try:
            km, km_err = kernel_ms(torch, bam, pinned), None
        except Exception as e:  # noqa: BLE001 -- the wall and phase times stand without the trace
            km, km_err = None, repr(e)
        ph = {("on" if f else "off"): {k: float(np.median([p[k] for p in phases[f]])) * 1e3 for k in phases[f][0]} for f in (False, True)}
        w = {("on" if f else "off"): stats(wall[f]) for f in (False, True)}
        floor_ms = ing["inflated_bytes"] / (res["hbm_copy_rate_GBps"] * 1e9) * 1e3
        r = {"records": n_rec, "bam_bytes": int(raw.size), "inflated_bytes": ing["inflated_bytes"], "bgzf_blocks": ing["bgzf_blocks"],
             "wall": w, "device_phase_ms_median": ph,
             "added_wall_median": w["on"]["median_ms"] / w["off"]["median_ms"] - 1.0, "added_wall_min": w["on"]["min_ms"] / w["off"]["min_ms"] - 1.0,
             "inflate_phase_delta_ms": ph["on"]["inflate"] - ph["off"]["inflate"],
             "hbm_floor_ms": floor_ms}
        if km_err:
            r["profiler_error"] = km_err
        if km:
            r["crc_kernel_ms"], r["crc_kernel_calls_profiled"] = km
            r["crc_kernel_GBps"] = ing["inflated_bytes"] / (km[0] * 1e-3) / 1e9
            r["hbm_floor_over_kernel"] = floor_ms / km[0]
        res[order] = r
        del pinned, raw
        torch.cuda.empty_cache()
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
