"""Cost of one BAM ingested by W GPUs (bam.ingest_bam_sharded) against the single-GPU ingest (bam.ingest_bam), on a synthetic
sample of bench.py's shape (synth.write_bam_fast, K = 4 alignments per read, read length 150), in both file orders.

  python profiles/tools/sharded_ingest_cost.py gen --dir D [--reads 8000000]        # writes D/name.bam, D/coord.bam
  torchrun --nproc-per-node W profiles/tools/sharded_ingest_cost.py run --dir D --out J  # adds the W-rank rows to J

Per file and W: the maximum over ranks of every phase (plan = block search + verification, read = disk -> page-locked memory,
inflate = H2D + hardware inflate (read included), chain, partition, exchange, back half; host wall clock, each phase ends with the
device idle), the bytes that crossed between ranks and their rate over the slowest rank's exchange, records/s over the slowest rank's
wall time, each rank's device memory in use after the call (the ingest's workspace cache keeps its high-water mark), the ranks'
record and inflated-byte shares, and parity: every rank's score stream, its owned contigs' pileup record counts and plane words, and
the ranks' summed n_dropped against the single-GPU ingest of the same file on the same device.  The card's name and power limit are
recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, ROOT)


def gen(args):
    import torch
    import bench
    from metamlst_b200 import synth
    os.makedirs(args.dir, exist_ok=True)
    ns = argparse.Namespace(reads=args.reads, read_len=150, k=4, alleles=1024)
    db = bench.make_db(ns)
    for order in ("name", "coord"):
        cores = bench.gen_cores(db, ns, torch.device("cuda", 0), None, seed=1002, n_reads=args.reads)
        raw = synth.write_bam_fast(db, cores, order=order, align_records=True)
        del cores
        raw.tofile(os.path.join(args.dir, order + ".bam"))
        print(order, raw.size, "bytes", flush=True)
        del raw
        torch.cuda.empty_cache()


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30).stdout.decode().strip()
    except Exception:  # noqa: BLE001
        pl = "not measured"
    return {"name": name, "power_limit": pl}


def run(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from metamlst_b200 import api, bam
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", local)
    rows = {}
    for order in ("name", "coord"):
        path = os.path.join(args.dir, order + ".bam")
        free0, total = torch.cuda.mem_get_info(dev)
        st = bam.ingest_bam_sharded(path, local, want_qhash=False)       # warm-up: driver entry points, workspace
        del st
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        st = bam.ingest_bam_sharded(path, local, want_qhash=False)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        free1, _ = torch.cuda.mem_get_info(dev)
        sh = st.shard
        mine = {"wall": wall, "seconds": sh["seconds"], "records_parsed": sh["records_parsed"], "records_received": sh["records_received"],
                "bytes_sent": sh["bytes_sent"], "bytes_received": sh["bytes_received"], "inflated_bytes": st.ingest_stats["inflated_bytes"],
                "compressed_bytes": st.ingest_stats["compressed_bytes"], "device_bytes_in_use_after": int(total - free1),
                "device_bytes_in_use_before": int(total - free0)}
        # the bytes this rank sent to other ranks (what an all-to-all moves between GPUs)
        # parity against the single-GPU ingest of the whole file, on this device
        whole = bam.ingest_bam(path, local, want_qhash=False)
        loc = api.AlleleIndex(whole.ref_names).locus_of
        owner = torch.as_tensor((np.asarray(loc, dtype=np.int64) % world).astype(np.int64), device=dev)
        keep = owner[whole.tid.long()] == rank
        oi = whole.orig_idx if whole.orig_idx is not None else torch.arange(whole.tid.shape[0], dtype=torch.int32, device=dev)
        same = (torch.equal(st.tid, whole.tid[keep]) and torch.equal(st.as0, whole.as0[keep]) and torch.equal(st.xm3, whole.xm3[keep])
                and torch.equal(st.qlen, whole.qlen[keep]) and torch.equal(st.orig_idx, oi[keep]))
        cs_w, cs_s = np.diff(whole.contig_start.astype(np.int64)), np.diff(st.contig_start.astype(np.int64))
        own_t = (np.asarray(loc, dtype=np.int64) % world) == rank
        same = same and bool(np.array_equal(cs_s[own_t], cs_w[own_t]) and not cs_s[~own_t].any())
        mine["parity"] = bool(same)
        mine["n_dropped"] = int(st.n_dropped)
        mine["whole_n_dropped"] = int(whole.n_dropped)
        mine["whole_records"] = int(whole.tid.shape[0])
        del whole, st
        torch.cuda.synchronize()
        got = [None] * world
        dist.all_gather_object(got, mine)
        if rank == 0:
            phases = sorted(got[0]["seconds"])
            xbytes = sum(g["bytes_sent"] for g in got)
            n = got[0]["whole_records"]
            rows[order] = {
                "records": n,
                "wall_seconds_max": max(g["wall"] for g in got),
                "records_per_s": n / max(g["wall"] for g in got),
                "phase_seconds_max": {p: max(g["seconds"].get(p, 0.0) for g in got) for p in phases},
                "exchange_bytes_all_ranks": xbytes,
                "exchange_GBps": xbytes / max(g["seconds"]["exchange"] for g in got) / 1e9,
                "device_bytes_in_use_after_per_rank": [g["device_bytes_in_use_after"] for g in got],
                "device_bytes_in_use_before_per_rank": [g["device_bytes_in_use_before"] for g in got],
                "records_parsed_per_rank": [g["records_parsed"] for g in got],
                "records_received_per_rank": [g["records_received"] for g in got],
                "inflated_bytes_per_rank": [g["inflated_bytes"] for g in got],
                "compressed_bytes_per_rank": [g["compressed_bytes"] for g in got],
                "parity_every_rank": all(g["parity"] for g in got),
                "n_dropped_sum_equals_whole": sum(g["n_dropped"] for g in got) == got[0]["whole_n_dropped"],
            }
            print(json.dumps({"W": world, order: rows[order]}), flush=True)
    if rank == 0:
        data = json.load(open(args.out)) if os.path.exists(args.out) else {}
        data.setdefault("card", card())
        data.setdefault("how", __doc__.strip().split("\n\n")[-1])
        data.setdefault("runs", {})["W=%d" % world] = rows
        json.dump(data, open(args.out, "w"), indent=1)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["gen", "run"])
    ap.add_argument("--dir", required=True)
    ap.add_argument("--reads", type=int, default=8_000_000, help="reads (x 4 records)")
    ap.add_argument("--out", default="sharded_ingest_cost.json")
    args = ap.parse_args()
    gen(args) if args.mode == "gen" else run(args)


if __name__ == "__main__":
    main()
