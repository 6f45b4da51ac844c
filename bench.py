#!/usr/bin/env python3
"""bench.py -- aligned reads/s through score + pileup + consensus (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--reads R --alleles A] [--dump-outputs DIR]

Workload (N=1): BASELINE.json configs[1] -- one sample of 10 M x 150 bp reads, K=4 alignments per read (40 M BAM
records, coordinate-sorted), against the synthetic E. coli + S. aureus + K. pneumoniae schemes (21 loci x 1024
alleles).  A "step" is one full pass of the hot path over that sample.  For N>1 every rank owns the records of a
disjoint set of loci (contig-aligned shards, 10 M reads each: weak scaling) and the integer tables are all-reduced.

  value     : records/s with the packed streams already resident in HBM (CUDA events, max over ranks)
  e2e       : the same pass through the host-buffer C-ABI (mmlst_sample: one call per sample) from pinned host memory,
              host<->device copies inside the timed region; both streams cross PCIe as DEFLATE blocks inflated by the
              hardware decompression engine; several samples in flight (api.SampleLanes), one at a time beside it
  roofline  : dominant kernel of the step against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline / --impl reference : the C port of the oracle on the host cores, on the WHOLE sample
The headline mode is the reference's own semantics (pysam max_depth = 8000, "parity mode"); the same sample without
the htslib depth cap (full 1.5 G-increment histogram) is reported under "uncapped".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=48, help="timed passes (a pass is ~40 us: the default keeps every cohort lane busy for several passes)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU")
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--alleles", type=int, default=1024, help="alleles per locus")
    ap.add_argument("--k", type=int, default=4, help="alignments per read")
    ap.add_argument("--pileup-impl", type=int, default=0)
    ap.add_argument("--no-extras", action="store_true", help="skip uncapped / hamming / cpu baseline extras")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph replay of the pass")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the full-workload comparison with the C port of the oracle after the timed region")
    ap.add_argument("--ingest-reads", type=int, default=2_000_000, help="reads of the BAM the `ingest` leg starts from (x K records; 0 = skip the leg)")
    ap.add_argument("--only-ingest", action="store_true", help="run only the BAM ingest leg (profiling aid)")
    ap.add_argument("--only-hamming", action="store_true", help="run only the configs[4] Hamming sweep (profiling aid)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "gather", "allreduce"],
                    help="N>1: 'p2p' = owner mode, result blocks stored into the peers' memory over NVLink by our own kernels; 'gather' = owner mode, "
                         "one NCCL all-gather of result blocks per pass; 'allreduce' = partial score/count tensors all-reduced with NCCL")
    ap.add_argument("--lanes", type=int, default=0, help="streams that consecutive passes alternate on (cohort mode: the latency-bound tail of a "
                    "pass overlaps the scoring kernels of the next ones); 1 = strictly serial passes; 0 = default: 6 (r1t, N=1: 4 lanes 1.05e12, 6 lanes "
                    "1.17e12, 8 lanes 1.18e12 records/s; r1u, N=2: 2 lanes 1.49e12, 6 lanes 2.30e12)")
    ap.add_argument("--no-qc", action="store_true", help="score stream in the 5 B/record run-length form (explicit len(SEQ) per record) even when every "
                    "256-record chunk is uniform")
    ap.add_argument("--score-variant", default="default", choices=["default", "0", "1", "2", "3", "4", "5", "6", "auto"],
                    help="form of the run-length score kernel (mmlst_set_score_variant): 0 registers, 1 registers + software pipeline, 2 shared-memory "
                         "ring fed by TMA bulk copies; 'default' = the library's; 'auto' = time all three on the workload first and keep the fastest")
    ap.add_argument("--score-l2-hints", default="default", choices=["default", "0", "1"], help="ring forms of the score kernel: L2 residency hints "
                    "(mmlst_set_score_l2_hints)")
    ap.add_argument("--e2e-cover", type=float, default=1.0, help="fraction of as0[] / xm3[] shipped as DEFLATE blocks in the `e2e` leg (the rest plain; r3e: with several "
                    "samples in flight the whole arrays compressed is fastest -- 1.16 ms per sample at 1.0 against 1.24 at 0.95 and 1.32 at 0.9)")
    ap.add_argument("--e2e-level", type=int, default=6, help="zlib level of the DEFLATE blocks of the `e2e` leg (6: 0.41 bytes per record for as0 + 6 xm3 and xm3 "
                    "against 0.49 at level 3, for twice the preparation time)")
    ap.add_argument("--e2e-plain-pileup", action="store_true", help="`e2e` leg: ship the chosen contigs' pileup records plain instead of as DEFLATE blocks")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="samples in flight in the `e2e` leg (api.SampleLanes); 1, 2 and 3 are always timed and reported beside it")
    ap.add_argument("--max-depth", type=int, default=8000, help="htslib pileup depth cap of the main workload (0 = uncapped; profiling aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed passes, write what the last one returned (chosen alleles, "
                    "consensus, holes, SNPs, read counters) as DIR/<name>.npy in float64, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


ORGS = ("ecoli", "saureus", "kpneumoniae")
PROPS = (0.5, 0.3, 0.2)
PARAMS = dict(minscore=80, max_xM=5, min_read_len=50, penalty=100)


def ncu_traffic(kernel):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(kernel, {}).get("dram_bytes_per_launch")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML (nvidia_ml_py) every 10 ms while the GPU is under load:
    started before the warm-up, stopped after the timed region (B200_PROFILING.md recipe, same counters)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.reasons, self.max_sm = [], set(), None
        self.period = 0.01
        self._stop = threading.Event()
        self._t = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            return
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                 "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

        def loop():
            while not self._stop.is_set():
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:  # noqa: BLE001
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:  # noqa: BLE001
                    pass
                time.sleep(self.period)
        self._t = threading.Thread(target=loop, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=1)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "how": "NVML every 10 ms from warm-up start to the end of the device-timed region, every 100 ms during the host-timed "
                                                "`e2e` region (an NVML query every 10 ms slows the host-side enqueue of the copies it times)"}


def make_db(args):
    from metamlst_b200 import synth
    return synth.make_db(ORGS, alleles_per_locus=args.alleles, n_profiles=2048, seed=1002)


def gen_cores(db, args, device, locus_subset=None, seed=1002, n_reads=None, chunk=1_000_000):
    """The reads of one synthetic sample as synth.gen_core chunks (deterministic in (seed, device kind))."""
    from metamlst_b200 import synth
    n_reads = n_reads or args.reads
    cores = []
    for i, c0 in enumerate(range(0, n_reads, chunk)):
        core = synth.gen_core(db, min(chunk, n_reads - c0), args.read_len, seed=seed * 1000 + i, K=args.k, org_props=PROPS,
                              device=device, strain_seed=1002, locus_subset=locus_subset)
        # keep only what the packers need
        cores.append({k: core[k] for k in ("L", "K", "bases", "qual", "rtype", "a_split", "rows", "start", "flag", "AS", "xm")})
        del core
    return cores


def gen_streams(db, args, device, max_depth, locus_subset=None, seed=1002, n_reads=None, chunk=1_000_000, want_qhash=False):
    from metamlst_b200 import devpack
    import torch
    cores = gen_cores(db, args, device, locus_subset, seed, n_reads, chunk)
    st = devpack.pack_cores(db, cores, 20, max_depth, want_qhash=want_qhash)
    n_ops = sum(int((c["rtype"] != 0).sum()) * 2 for c in cores) * args.k  # extra CIGAR ops beyond 1 per record
    del cores
    if device != "cpu":
        torch.cuda.empty_cache()
    return st, n_ops


def cpu_workload(db, args, device, locus_subset=None, seed=1002, n_reads=None):
    """The SAME sample (same generator, seeds and record order) unpacked on the host for the C port of the oracle."""
    import torch
    from oracle import cpu_path
    cores = gen_cores(db, args, device, locus_subset, seed, n_reads)
    w = cpu_path.workload_from_cores(db, cores)
    del cores
    if device != "cpu":
        torch.cuda.empty_cache()
    return w


def pileup_alg_bytes(st, tids, L):
    """SURVEY.md 8d: per admitted record on a chosen contig 8 + 4 n_ops + L/2 bytes; + 21.25 B per column."""
    recs = sum(int(st.contig_start[t + 1] - st.contig_start[t]) for t in tids)
    cols = sum(int(st.ref_lens[t]) for t in tids)
    return recs * (8 + 4 * 1.22 + L / 2.0) + cols * 21.25, recs  # 1.22 = mean CIGAR ops of the generator (89 % 1 op, 11 % 3)


def event_ms(pairs):
    return [a.elapsed_time(b) for a, b in pairs]


def dump_outputs(out_dir, result, total_reads, ignored_reads, name_to_tid):
    """One pass's result ({species: [(contig, consensus, holes, snps)]} in the reference's dict order, totalReads, ignoredReads)
    as float64 arrays, one entry per chosen locus in that order; every value is an integer well below 2**53, so nothing is rounded."""
    rows = [(c, s, h, n) for sp in result for (c, s, h, n) in result[sp]]
    arrays = {"allele": [name_to_tid[c] for c, _s, _h, _n in rows],
              "consensus_len": [len(s) for _c, s, _h, _n in rows],
              "consensus": np.frombuffer("".join(s for _c, s, _h, _n in rows).encode("latin-1"), np.uint8),
              "holes": [h for _c, _s, h, _n in rows],
              "snps": [n for _c, _s, _h, n in rows],
              "reads": [total_reads, ignored_reads]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


# ----------------------------------------------------------------------------------------------------------------
def cpu_port_run(w, args, threads, steps=1, warmup=0):
    """The oracle's C port (oracle/cpu_path.py over oracle/c) on the host cores over the WHOLE sample `w`: score of every record,
    selection, htslib depth-cap simulation over every record of the chosen contigs, pileup of the admitted ones, consensus --
    the regime of the GPU arm (same records, same cap).  Returns (records/s, seconds per step, last result, description)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cpu_path
    pool = ThreadPoolExecutor(threads) if threads > 1 else None
    kw = dict(minscore=PARAMS["minscore"], max_xM=PARAMS["max_xM"], min_read_len=PARAMS["min_read_len"], penalty=PARAMS["penalty"],
              max_depth=args.max_depth or None, threads=threads, pool=pool)
    for _ in range(warmup):
        cpu_path.run(w, **kw)
    phases = {}
    t0 = time.perf_counter()
    for _ in range(steps):
        res = cpu_path.run(w, **kw)
        for k, v in res["seconds"].items():
            phases[k] = phases.get(k, 0.0) + v / steps
    dt = (time.perf_counter() - t0) / steps
    if pool is not None:
        pool.shutdown()
    sample = ("the WHOLE sample of `config.workload` (%d records; %d on the chosen contigs walked by the htslib depth-cap simulation, %d of them "
              "admitted and piled up), C port of the oracle (oracle/c/mlst_oracle.c via oracle/cpu_path.py), %d thread(s); seconds per step: "
              "score %.4f, select %.4f, depth cap + pileup + consensus %.4f" % (
                  w.n, res["chosen_contig_records"], res["piled_records"], threads, phases["score"], phases["select"], phases["depthcap_pileup_consensus"]))
    return w.n / dt, dt, res, sample, phases


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference itself is pure Python over pysam / samtools /
    Biopython, none of which exist on the box (DESIGN.md section 2), so this arm times the C port of its restatement -- a FASTER
    stand-in -- on all host threads over the same full sample the GPU arm types (same generator, seeds, depth cap)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    db = make_db(args)
    threads = os.cpu_count() or 1
    dev = "cuda:%d" % int(os.environ.get("LOCAL_RANK", "0")) if torch.cuda.is_available() else "cpu"
    w = cpu_workload(db, args, dev)
    steps = max(1, args.steps)
    rate, dt, res, sample, phases = cpu_port_run(w, args, threads, steps=steps, warmup=min(max(args.warmup, 0), 2))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res["result"], int(res["counters"][0]), int(res["counters"][1]), {n: i for i, n in enumerate(db.ref_names())})
    cfg = workload_config(args, 1)
    line = {"impl": "reference", "metric": "aligned reads/s (score+pileup+consensus)", "value": rate, "unit": "records/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32/u8", "data": "synthetic",
            "config": {"workload": cfg["workload"], "mode": cfg["mode"],
                       "arm": "host cores only: C port of the oracle, %d threads, records unpacked in host memory (score: %d record ranges; pileup: "
                              "one chosen contig per task)" % (threads, threads)},
            "gpu_launches": 0, "seconds_by_phase": phases,
            "cpu_baseline": {"value": rate, "unit": "records/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "the reference itself (pure Python over pysam/samtools) cannot run on this box; this is the C port of its restatement (oracle/c), "
                    "a faster stand-in; the Python reference measured in the build container: profiles/r1_reference_python_timing.json (4.0e3 records/s)"}
    emit(line)


def workload_config(args, world):
    return {"workload": "configs[1]: single sample, %d x %d bp reads, K=%d alignments/read (%d BAM records per GPU), coordinate-sorted; "
                        "E. coli + S. aureus + K. pneumoniae synthetic schemes, 21 loci x %d alleles" % (args.reads, args.read_len, args.k, args.reads * args.k, args.alleles),
            "mode": ("parity (htslib max_depth %d, minqual 20, minscore 80, max_xM 5)" % args.max_depth) if args.max_depth else "uncapped (no depth cap; NOT the reference's semantics)",
            "sharding": "replica" if world == 1 else ("contig-aligned: each rank owns the records of a disjoint locus set; " + (
                "owner mode, result blocks stored straight into every peer's memory over NVLink (csrc/exchange.cu: publish + await kernels, no NCCL "
                "call inside the pass)" if args.exchange == "p2p" else
                "owner mode, ONE NCCL all-gather of the per-rank result blocks per pass" if args.exchange == "gather" else
                "all-reduce SUM(sum_as,n_hit,counters) MIN(first_idx) SUM(counts)")),
            "schedule": ("cohort mode: consecutive passes alternate over %d streams, so the latency-bound tail of pass i (selection, capped pileup, "
                         "consensus%s) runs under the HBM-bound scoring kernel of pass i+1; every pass is complete (own tables, own D2H) inside the timed "
                         "region; strictly serial passes: serial_ms_per_step" % (args.lanes, ", the exchange" if world > 1 else ""))
            if args.lanes > 1 else "serial passes on one stream",
            "l2": "consecutive passes type two different samples of this shape alternately (a cohort): their score streams together (2 x %d MB in the "
                  "3 B/record form, 2 x %d MB in the 5 B form) exceed the 126 MB L2, so every pass streams its input from HBM; per-kernel timings: score "
                  "alternates the two samples back to back, select/pileup/consensus are timed one launch at a time after rewriting a 256 MB buffer "
                  "(L2 flush)" % (args.reads * args.k * 3 // 1000000, args.reads * args.k * 5 // 1000000)}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank's host threads (and, by first touch, its page-locked buffers) on the NUMA node the GPU hangs off: with 8 ranks pushing
    host buffers at PCIe speed, cross-socket traffic was what held e2e scaling back in round 1.  Best effort; returns a description."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return "numa_node -1 (single node)"
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "node %d, %d cpus" % (node, len(allowed))
        return "node %d has no allowed cpu" % node
    except Exception as e:  # noqa: BLE001
        return "unbound (%r)" % (e,)


_REAL_STDOUT = None


def protect_stdout():
    """Everything any library prints to fd 1 (NCCL's version banner, ...) goes to stderr; the ONE JSON line is written to
    the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    (_REAL_STDOUT or sys.stdout).write(json.dumps(line) + "\n")
    (_REAL_STDOUT or sys.stdout).flush()


def main():
    args = parse()
    protect_stdout()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    from metamlst_b200 import api, native, pipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.lanes <= 0:
        args.lanes = 6
    numa = bind_to_gpu_numa_node(local) if world > 1 else "not bound (one rank)"
    torch.cuda.set_device(local)
    device = "cuda:%d" % local
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device(device))
    native.lib()  # fail loudly if the CUDA library is missing
    if args.score_variant in ("0", "1", "2", "3", "4", "5", "6"):
        native.lib().mmlst_set_score_variant(int(args.score_variant))
    if args.score_l2_hints in ("0", "1"):
        native.lib().mmlst_set_score_l2_hints(int(args.score_l2_hints))
    score_variant = native.lib().mmlst_set_score_variant(-1)
    score_hints = native.lib().mmlst_set_score_l2_hints(-1)
    peak, peak_src = peaks()
    if args.only_hamming:
        emit({"hamming": extra_hamming(device, peak)})
        return
    if args.only_ingest:
        emit({"ingest": extra_ingest(make_db(args), args, device)})
        return

    db = make_db(args)
    index = api.AlleleIndex(db.ref_names())
    n_loci = len(db.locus_names)
    subset = None if world == 1 else [l for l in range(n_loci) if l % world == rank]
    st, _ = gen_streams(db, args, device, args.max_depth or None, subset, seed=1002 + rank)
    R_local = int(st.tid.shape[0])
    if world > 1 and args.exchange == "p2p":
        # peer-mapped memory needs P2P access between the GPUs of the box: probe it once, and let every rank agree
        ok = 1
        try:
            import torch.distributed._symmetric_memory as symm
            probe = symm.empty(4096, dtype=torch.uint8, device=device)
            symm.rendezvous(probe, torch.distributed.group.WORLD)
        except Exception as e:  # noqa: BLE001
            sys.stderr.write("peer-mapped memory unavailable (%r): using the NCCL all-gather form\n" % (e,))
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
        if int(flag.item()) == 0:
            args.exchange = "gather"
    # consecutive passes type DIFFERENT samples of the same shape (a cohort): two samples' score streams together exceed
    # the 126 MB L2 whatever the stream form, so no pass finds its input cached by the previous one
    n_samples = max(2, args.lanes)
    sts = [st] + [gen_streams(db, args, device, args.max_depth or None, subset, seed=1002 + rank + 100 * l)[0] for l in range(1, n_samples)]
    assert all(int(x.tid.shape[0]) == R_local for x in sts)
    if args.no_qc:
        for x in sts:
            x.chunk_qlen = None
    pipes = [pipeline.DevicePipeline(x, index, db.row_seq, impl=args.pileup_impl, idx_base=rank * R_local, exchange=args.exchange, **PARAMS) for x in sts]
    pipe = pipes[0]

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    variants_ms = None
    if args.score_variant == "auto" and pipe.use_runs:
        # every form on this workload (equal tables asserted), fastest kept for everything that follows; with N>1 the ranks agree on rank 0's choice
        variants_ms = pipe.time_score_variants(20, alt=pipes[1])
        if os.environ.get("MMLST_BENCH_SCALING"):  # profiling aid (profiles/run_p.sh): launch time at 1/1, 1/2, 1/4 of the stream, per form
            for key in sorted(variants_ms):
                native.lib().mmlst_set_score_variant(int(key[0]))
                native.lib().mmlst_set_score_l2_hints(1 if key.endswith("h") else 0)
                sys.stderr.write("score form %s, records 1/1 1/2 1/4: %r\n" % (key, pipe.time_score_half(20, alt=pipes[1])))
        best = min(variants_ms, key=variants_ms.get)
        pick = torch.tensor([int(best[0]), 1 if best.endswith("h") else 0], dtype=torch.int32, device=device)
        if world > 1:
            torch.distributed.broadcast(pick, 0)
        score_variant, score_hints = int(pick[0].item()), int(pick[1].item())
        native.lib().mmlst_set_score_variant(score_variant)
        native.lib().mmlst_set_score_l2_hints(score_hints)
    results = []
    for p in pipes:
        for _ in range(max(args.warmup, 3)):
            r = p.step()
        results.append(r)
    result = results[0]
    use_graph = not args.no_graph
    if use_graph:
        try:
            for p, r in zip(pipes, results):
                p.capture()
                assert p.step_graph() == r, "graph replay differs from the eager pass"
        except Exception as e:  # noqa: BLE001
            sys.stderr.write("CUDA graph capture unavailable (%r): timing the eager pass\n" % (e,))
            use_graph = False
    if not use_graph:
        for p in pipes:
            p.graph = None
    barrier()
    for p in pipes:
        p.launches = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    prof = bool(os.environ.get("MMLST_CUDA_PROFILER"))  # `ncu --profile-from-start off`: capture the timed steps only
    if prof:
        torch.cuda.profiler.start()
    # K passes queued back to back (each one ends with its D2H into the pinned output block); the host parses the
    # result after the timed region -- the way a cohort is typed.  Per-pass latency WITH a host sync is reported too.
    e0.record()
    for i in range(args.steps):
        pipes[i % n_samples].enqueue_step()
    e1.record()
    barrier()
    outs_serial = [p.collect() for p in pipes]
    out = outs_serial[0]
    assert outs_serial == results, "results changed between steps"
    k = (args.steps - 1) % n_samples
    last = (outs_serial[k], pipes[k].total_reads, pipes[k].ignored_reads)
    serial_ms = e0.elapsed_time(e1) / args.steps
    serial_launches = sum(p.launches for p in pipes)
    # the same serial passes alternating between TWO samples only: both score streams (2 x 121 MB) still exceed the L2 and are streamed from HBM every
    # pass (they are read evict-first), but a sample's tail inputs -- selection tables, the 40 MB of depth-capped pileup records -- may survive in the L2
    # from its previous pass: the regime of a device that keeps typing against a warm working set (profiles/r3j_hints*_l1.json)
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(4):
        pipes[i % 2].enqueue_step()
    e2.record()
    for i in range(args.steps):
        pipes[i % 2].enqueue_step()
    e3.record()
    barrier()
    assert [p.collect() for p in pipes[:2]] == results[:2], "results changed between steps"
    serial2_ms = e2.elapsed_time(e3) / args.steps
    lanes = None
    if args.lanes > 1:
        # cohort mode: passes alternate over `lanes` streams, each lane with its own tables / output block / graph and, with
        # N>1, its own NCCL communicator (collectives of different lanes may be in flight together)
        groups = [torch.distributed.new_group(list(range(world))) if world > 1 and args.exchange != "p2p" else None for _ in range(args.lanes)]
        lanes = pipeline.CohortLanes(lambda lane: pipeline.DevicePipeline(sts[lane % n_samples], index, db.row_seq, impl=args.pileup_impl,
                                                                          idx_base=rank * R_local, exchange=args.exchange, group=groups[lane], **PARAMS), args.lanes)
        want = [results[lane % n_samples] for lane in range(args.lanes)]
        assert lanes.warm_and_capture(graph=use_graph) == want, "a cohort lane disagrees with the serial pass"
        for i in range(2 * args.lanes):  # warm the overlapped schedule itself
            lanes.enqueue(i)
        assert lanes.collect() == want
        for p in lanes.pipes:
            p.launches = 0
        barrier()
        e0.record()
        lanes.fork(e0)
        for i in range(args.steps):
            lanes.enqueue(i)
        lanes.join()
        e1.record()
        barrier()
        outs_lanes = lanes.collect()
        assert outs_lanes == want, "cohort-mode results differ from the serial pass"
        k = (args.steps - 1) % args.lanes
        last = (outs_lanes[k], lanes.pipes[k].total_reads, lanes.pipes[k].ignored_reads)
    if prof:
        torch.cuda.profiler.stop()
    assert out == result, "results changed between steps"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last, index.name_to_tid)
    launches = lanes.launches if lanes is not None else serial_launches
    # per-kernel durations: 20 back-to-back launches of each kernel of the same pass between two CUDA events on the
    # launching stream (events are not graph-capturable; a single launch would carry the event/launch gap)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    kms = pipe.time_kernels(20, alt=pipes[1], flush=flush)
    del flush
    # the other forms of the score kernel on the same two samples (same tables out, checked), for the record
    if variants_ms is None:
        variants_ms = {str(score_variant) + ("h" if score_hints and score_variant >= 2 else ""): kms["score"]}
        if not args.no_extras and pipe.use_runs:
            variants_ms = pipe.time_score_variants(20, alt=pipes[1])
            native.lib().mmlst_set_score_variant(score_variant)
            native.lib().mmlst_set_score_l2_hints(score_hints)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        assert (pipe.step_graph() if use_graph else pipe.step()) == result
    lat_ms = (time.perf_counter() - t0) / 10 * 1e3
    ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t.item())
    R_total = R_local * world
    tids = [index.name_to_tid[c] for sp in out for (c, _s, _h, _n) in out[sp]]
    # bytes the score kernel has to read: the run-length form stores the allele id per run (5 B / record + 8 B / run +
    # 4 B / 256-record chunk); SURVEY.md 8d's 9 B / record assumed an explicit 4-byte id per record (kept as a fallback form)
    if pipe.use_qc:
        score_bytes = 3.0 * R_local + 8.0 * int(st.run_tid.shape[0]) + 6.0 * int(st.chunk_run.shape[0])
    elif pipe.use_runs:
        score_bytes = 5.0 * R_local + 8.0 * int(st.run_tid.shape[0]) + 4.0 * int(st.chunk_run.shape[0])
    else:
        score_bytes = 9.0 * R_local
    pb, precs = pileup_alg_bytes(st, [t for t in tids if st.contig_start[t + 1] > st.contig_start[t]], args.read_len)
    rooflines = {
        "score": {"bound": "hbm", "achieved": score_bytes / kms["score"] / 1e6, "peak": peak, "unit": "GB/s", "frac": score_bytes / kms["score"] / 1e6 / peak,
                  "traffic": ncu_traffic("score_runs_qc" if pipe.use_qc else "score_runs" if pipe.use_runs else "score") if args.reads == 10_000_000 and args.k == 4 else None,
                  "ms": kms["score"], "algorithmic_bytes": score_bytes, "kernel_form": score_variant, "l2_hints": score_hints, "ms_by_kernel_form": variants_ms,
                  "stream_form": "run-length + len(SEQ) per 256-record chunk: as0 i16 + xm3 u8 per record, allele id per run (3 B/record; lossless: every "
                                 "chunk of this sample has one read length; SURVEY 8d's explicit form is 9 B/record)" if pipe.use_qc else
                                 "run-length: as0 i16 + xm3 u8 + qlen u16 per record, allele id per run (5 B/record; SURVEY 8d's explicit-id form is 9 B/record)"
                  if pipe.use_runs else "explicit allele id per record (9 B/record)"},
        "pileup_parity": {"bound": "hbm", "achieved": pb / kms.get("pileup", float("inf")) / 1e6, "peak": peak, "unit": "GB/s",
                          "frac": pb / kms.get("pileup", float("inf")) / 1e6 / peak, "traffic": None, "ms": kms.get("pileup"),
                          "algorithmic_bytes": pb, "records": precs},
        "consensus": {"ms": kms.get("consensus")},
    }
    dominant = max(("score", "pileup_parity"), key=lambda k: rooflines[k]["ms"] or 0)
    line = {"metric": "aligned reads/s (score+pileup+consensus)", "value": R_total / (ms / 1e3), "unit": "records/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32/u8 (integer bit-plane arithmetic)", "data": "synthetic",
            "config": workload_config(args, world), "clocks": None, "gpu_launches": launches,
            "roofline": dict(rooflines[dominant], kernel=dominant, peak_source=peak_src), "rooflines": rooflines,
            "kernel_ms_per_step": kms, "records_per_gpu": R_local, "cuda_graph": use_graph,
            "serial_ms_per_step": serial_ms, "serial_ms_per_step_two_samples": serial2_ms, "lanes": args.lanes if lanes is not None else 1,
            "non_kernel_ms_per_step": serial_ms - sum(kms.values()), "latency_ms_per_step_with_host_sync": lat_ms}

    # ---- end to end through the host-buffer C-ABI (pinned host memory -> results on the host), every rank on its own shard;
    # with N>1 the ranks' results are all-gathered inside the timed region (each rank owns whole loci)
    soa = st.to_host(pinned=True)
    t0 = time.perf_counter()
    # once per sample, like the unpacking: as0[] / xm3[] as DEFLATE blocks, inflated on the device by the hardware engine; the last tenth of each
    # array stays plain and rides the bus while the engine (the slower of the two on this data) drains its queue (profiles/r2z_e2e_sweep.json)
    soa.deflate(level=args.e2e_level, cover=args.e2e_cover, pileup=not args.e2e_plain_pileup)
    z_coeff = int(soa.z_as_xm_coeff)
    t_deflate = time.perf_counter() - t0
    ctx = native.Context(local)

    e2e_words = 1 + 3 * n_loci + (int(np.sort(np.asarray(st.ref_lens))[::-1][:n_loci].sum()) + 3) // 4 + 4
    if world > 1:
        e2e_pin = torch.zeros(e2e_words * 4, dtype=torch.uint8).pin_memory()
        e2e_dev = torch.zeros(e2e_words * 4, dtype=torch.uint8, device=device)
        e2e_all = torch.zeros(world * e2e_words * 4, dtype=torch.uint8, device=device)

    sidx = api.SampleIndex(ctx, index, st.ref_lens, db.row_seq)
    e2e_mode = {"one_call": True}
    sampler.period = float(os.environ.get("MMLST_BENCH_E2E_SAMPLER_PERIOD", "0.1"))

    # (--nloci gate: 100 on one rank; a rank that owns a subset of the loci cannot apply it -- the owner of the merge would, as in pipeline.py)
    one_call_kw = dict(minscore=PARAMS["minscore"], max_xM=PARAMS["max_xM"], min_read_len=PARAMS["min_read_len"], penalty=PARAMS["penalty"],
                       nloci=100 if world == 1 else 0, impl=args.pileup_impl)

    def unpack_one_call(r):
        flat = [x for _sp, lst in r["species"] for x in lst]
        return r["tids"], [x[1] for x in flat], [x[2] for x in flat], [x[3] for x in flat]

    def e2e_step():
        if e2e_mode["one_call"]:
            # ONE library call per sample (mmlst_sample): score stream up + inflate, score, selection on the device, the chosen contigs' pileup records up,
            # pileup, consensus, results down
            ts, seqs, holes, snps = unpack_one_call(api.type_soa(sidx, soa, **one_call_kw))
        else:
            # the two seams as separate calls (mmlst_score -> host selection -> mmlst_pileup_consensus): the reference's own call structure
            cel_raw = api.score_soa_raw(ctx, soa, index, **{k: PARAMS[k] for k in ("minscore", "max_xM", "min_read_len")})
            chosen = api.fast_select(index, cel_raw[0], cel_raw[1], cel_raw[2], PARAMS["penalty"])
            ts = [t for _sp, tt in chosen for t in tt]
            seqs, holes, snps, _, _ = api.pileup_consensus(ctx, soa, ts, [db.row_seq(t) for t in ts], PARAMS["minscore"], PARAMS["max_xM"], 1, args.pileup_impl)
        return e2e_exchange(ts, seqs, holes, snps)

    def e2e_exchange(ts, seqs, holes, snps):
        mine = {index.ref_names[t]: (seqs[i], int(holes[i]), int(snps[i])) for i, t in enumerate(ts)}
        if world > 1:
            # every rank's result block to every rank: ONE fixed-size all-gather (NCCL) of [n | tid, holes, snps per locus | consensus bytes]
            blk = np.zeros(e2e_words * 4, np.uint8)
            w32 = blk.view(np.int32)
            w32[0] = len(ts)
            w32[1:1 + len(ts)] = ts
            w32[1 + n_loci:1 + n_loci + len(ts)] = holes[:len(ts)]
            w32[1 + 2 * n_loci:1 + 2 * n_loci + len(ts)] = snps[:len(ts)]
            cat = "".join(seqs).encode("latin-1")
            blk[(1 + 3 * n_loci) * 4:(1 + 3 * n_loci) * 4 + len(cat)] = np.frombuffer(cat, np.uint8)
            e2e_pin.numpy()[:] = blk
            e2e_dev.copy_(e2e_pin, non_blocking=True)
            torch.distributed.all_gather_into_tensor(e2e_all, e2e_dev)
            allb = e2e_all.cpu().numpy().reshape(world, -1)
            mine = {}
            for r in range(world):
                v32 = allb[r].view(np.int32)
                n = int(v32[0])
                off = (1 + 3 * n_loci) * 4
                for i in range(n):
                    t = int(v32[1 + i])
                    ln = int(st.ref_lens[t])
                    mine[index.ref_names[t]] = (allb[r][off:off + ln].tobytes().decode("latin-1"), int(v32[1 + n_loci + i]), int(v32[1 + 2 * n_loci + i]))
                    off += ln
        return ts, mine

    want_e2e = {c: (s_, h_, n_) for sp in out for (c, s_, h_, n_) in out[sp]}
    n_e2e = max(3, min(args.steps, 10))

    def time_e2e():
        for _ in range(2):
            ts_, r0 = e2e_step()
        assert r0 == want_e2e, "e2e result differs from the device-resident result"
        barrier()
        t0_ = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        return ts_, (time.perf_counter() - t0_) / n_e2e

    def time_e2e_lanes(n_lanes):
        """The same call with `n_lanes` samples in flight (api.SampleLanes: one context + host thread per lane, the cohort form of the host-buffer path).
        Every step still moves its own inputs up and its own results down inside the timed region; with N>1 the all-gather of every step's result
        blocks is issued by this thread in step order while later steps are already running."""
        sl = api.SampleLanes(local, index, st.ref_lens, db.row_seq, lanes=n_lanes)
        try:
            for r in sl.map([soa] * (2 * n_lanes), **one_call_kw):
                ts_, r0 = e2e_exchange(*unpack_one_call(r))
                assert r0 == want_e2e, "e2e (lanes) result differs from the device-resident result"
            n = max(8, n_e2e) * n_lanes
            barrier()
            t0_ = time.perf_counter()
            futs = [sl.submit(soa, **one_call_kw) for _ in range(n)]
            for f in futs:
                e2e_exchange(*unpack_one_call(f.result()))
            barrier()
            return (time.perf_counter() - t0_) / n
        finally:
            sl.close()

    # first the plain form (3 bytes per record cross PCIe), then the two seams as separate calls, then one call per sample with the compressed stream, one
    # sample at a time; then the headline: the same call with two samples in flight
    zb, zt, zp3 = soa.z_bytes, soa.z_table, (soa.zp_bytes, soa.zp_table, soa.zp_contig_block)
    soa.z_bytes = soa.z_table = soa.zp_bytes = soa.zp_table = soa.zp_contig_block = None
    ts_local, dt_plain = time_e2e()
    soa.z_bytes, soa.z_table = zb, zt
    soa.zp_bytes, soa.zp_table, soa.zp_contig_block = zp3
    e2e_mode["one_call"] = False
    ts_local, dt_seams = time_e2e()
    e2e_mode["one_call"] = True
    ts_local, dt_one = time_e2e()
    lanes_ms = {}
    for nl_ in sorted({1, 2, 3, args.e2e_lanes}):
        lanes_ms[nl_] = time_e2e_lanes(nl_)
    dt = lanes_ms[args.e2e_lanes]
    clocks = sampler.stop()
    line["clocks"] = clocks
    h2d_plain_score = ((3 * R_local + 6 * int(soa.chunk_run.shape[0]) if soa.chunk_qlen is not None else 5 * R_local + 4 * int(soa.chunk_run.shape[0])) +
                       8 * int(soa.run_tid.shape[0]) + 4) if soa.run_tid is not None else 9 * R_local
    z_cov = int((soa.z_table[:, 3] & np.uint64(0xffffffff)).sum())    # bytes of as0[] / xm3[] the DEFLATE blocks stand for; the rest travels plain
    h2d_score_zp = int(soa.z_bytes.shape[0]) + 3 * R_local - z_cov
    h2d = h2d_plain_score - 3 * R_local + h2d_score_zp + 32 * int(soa.z_table.shape[0]) if soa.z_bytes is not None else h2d_plain_score
    h2d += db.n_rows * 5
    proff = soa.p_row_off
    pileup_plain = int(sum((st.contig_start[t + 1] - st.contig_start[t]) * 16 for t in ts_local)) + \
        int(sum(int(proff[int(st.contig_start[t + 1])]) - int(proff[int(st.contig_start[t])]) for t in ts_local)) * 4
    if soa.zp_bytes is not None:   # the chosen contigs' DEFLATE blocks (compressed sizes from the block table)
        cb, zt_ = soa.zp_contig_block, soa.zp_table
        pileup_h2d = int(sum(int(((zt_[int(cb[t]):int(cb[t + 1]), 1] >> np.uint64(32)) & np.uint64(0x7fffffff)).sum()) for t in ts_local))
    else:
        pileup_h2d = pileup_plain
    h2d_plain_total_extra = pileup_plain - pileup_h2d   # what the plain / two-seam forms move on top (they ship records and rows uncompressed)
    h2d += pileup_h2d
    d2h_seams = db.n_rows * 16 + 16 + sum(int(st.ref_lens[t]) for t in ts_local) + 8 * len(ts_local)
    # one call: the selection block (header + chosen rows / species / column offsets), block sizes reported by the decompression engine, consensus, holes, snps
    d2h = (16 + 3 * n_loci + 1) * 4 + 4 * int(soa.z_table.shape[0]) + sum(int(st.ref_lens[t]) for t in ts_local) + 8 * n_loci
    h2d -= db.n_rows * 4    # locus_of[] is resident (mmlst_index_upload); allow[] still travels
    # what the box gives this path: every rank pulling from page-locked memory at once (GPUs share PCIe uplinks: profiles/r3q_h2d_probe_n8.json)
    bus_pin = torch.empty(128 << 20, dtype=torch.uint8).pin_memory()
    bus_dev = torch.empty(128 << 20, dtype=torch.uint8, device=device)
    for _ in range(2):
        bus_dev.copy_(bus_pin, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    t0_ = time.perf_counter()
    for _ in range(8):
        bus_dev.copy_(bus_pin, non_blocking=True)
    torch.cuda.synchronize()
    bus_s = time.perf_counter() - t0_
    barrier()
    del bus_pin, bus_dev
    lane_keys = sorted(lanes_ms)
    tt = torch.tensor([dt, float(h2d), float(d2h), dt_plain, dt_seams, dt_one] + [lanes_ms[k] for k in lane_keys] + [bus_s], dtype=torch.float64, device=device)
    h2d_rank_max = float(h2d)
    if world > 1:
        mx = tt.clone(); torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.SUM)
        dt = float(mx[0].item()); dt_plain = float(mx[3].item()); dt_seams = float(mx[4].item()); dt_one = float(mx[5].item())
        lanes_ms = {k: float(mx[6 + i].item()) for i, k in enumerate(lane_keys)}
        bus_s = float(mx[6 + len(lane_keys)].item()); h2d_rank_max = float(mx[1].item())
    bus_gbps = 8 * (128 << 20) / bus_s / 1e9
    line["e2e"] = {"value": R_total / dt, "unit": "records/s", "h2d_bytes_per_step": int(tt[1].item()), "d2h_bytes_per_step": int(tt[2].item()),
                   "ms_per_step": dt * 1e3, "timing": "host wall clock around the K synchronous C-ABI calls, barrier on both sides, max over ranks",
                   "call": "mmlst_sample (api.type_soa): one call per sample from pinned host buffers -- score stream up, score, selection on the device, pileup records "
                           "of the chosen contigs up, pileup, consensus, results down",
                   "schedule": "cohort mode, like `value`: %d samples in flight (api.SampleLanes: one context, stream and host thread per lane), so one sample's copies "
                               "ride the bus while another waits for its selection block or runs its pileup; every step's own H2D and D2H are inside the timed "
                               "region" % args.e2e_lanes,
                   "lanes": args.e2e_lanes,
                   "bus": {"h2d_GBps_per_gpu_all_ranks_copying": bus_gbps, "ms_per_step_at_that_rate": h2d_rank_max / bus_gbps / 1e6,
                           "what": "128 MB copies from page-locked memory, every rank at once, slowest rank: the GPUs of the box share PCIe uplinks, so the per-GPU rate "
                                   "falls as ranks are added (55 GB/s alone, 23 GB/s with 8: profiles/r3q_h2d_probe_n8.json); ms_per_step_at_that_rate = the largest "
                                   "rank's h2d bytes of a step at that rate, the floor of a bus-bound step"},
                   "ms_per_step_by_lanes": {str(k): lanes_ms[k] * 1e3 for k in sorted(lanes_ms)},
                   "one_at_a_time": {"value": R_total / dt_one, "unit": "records/s", "ms_per_step": dt_one * 1e3,
                                     "what": "the same call, strictly one sample after another on one context (single-sample latency)"},
                   "two_seam_calls": {"value": R_total / dt_seams, "unit": "records/s", "ms_per_step": dt_seams * 1e3,
                                      "what": "mmlst_score -> host selection -> mmlst_pileup_consensus, the reference's call structure, same compressed stream"},
                   "host_numa_binding": numa, "exchange": "one fixed-size NCCL all-gather of the per-rank result blocks" if world > 1 else "none (one rank)",
                   "stream_form": "the first %.0f %% of as0[] / xm3[] crosses PCIe as DEFLATE blocks and is inflated in HBM by the hardware decompression engine, slice by "
                                  "slice behind the copy, the rest plain (%.2f bytes per record in all instead of 3; the as0 blocks hold as0 + %d * xm3, the coefficient picked per sample, "
                                  "and a kernel subtracts it again after the inflate); deflating is part of preparing a sample "
                                  "(%.2f s here, host threads), like unpacking it; the chosen contigs' pileup records and plane rows cross as DEFLATE "
                                  "blocks too (%.1f MB instead of %.1f MB per sample)" % (100 * min(max(args.e2e_cover, 0.0), 1.0), h2d_score_zp / max(R_local, 1), z_coeff, t_deflate, pileup_h2d / 1e6, pileup_plain / 1e6),
                   "uncompressed": {"value": R_total / dt_plain, "unit": "records/s", "ms_per_step": dt_plain * 1e3,
                                    "h2d_bytes_per_step": int(tt[1].item()) + world * (3 * R_local - h2d_score_zp - 32 * int(soa.z_table.shape[0]) + h2d_plain_total_extra),
                                    "what": "the same call with the plain arrays (3 bytes per record cross PCIe)"}}
    ctx.close()
    del soa

    if not args.no_parity_check:
        # the benchmarked sample against the C port of the oracle, at FULL size (every rank on its own shard): score tables, chosen alleles,
        # consensus strings, holes, SNPs.  The same CPU pass is the `cpu_baseline` (rank 0, N=1): all host threads, and one thread.
        w = cpu_workload(db, args, device, subset, seed=1002 + rank)
        ncpu = os.cpu_count() or 1
        rate, dt_cpu, ref, sample, phases = cpu_port_run(w, args, ncpu, steps=1 if world > 1 else 3, warmup=0 if world > 1 else 1)
        pipe.reset_tables()
        pipe._score_call()
        torch.cuda.synchronize()
        checked = []
        if not (world > 1 and args.exchange == "allreduce"):
            assert np.array_equal(pipe.sum_as.cpu().numpy(), ref["sum_as"]), "sum_as differs from the C port on the full workload"
            assert np.array_equal(pipe.n_hit.cpu().numpy().view(np.uint32), ref["n_hit"]), "n_hit differs from the C port on the full workload"
            hit = ref["n_hit"] > 0
            assert np.array_equal(pipe.first_idx.cpu().numpy().view(np.uint32)[hit] - np.uint32(pipe.idx_base), ref["first_idx"][hit]), "first_idx differs"
            assert pipe.counters.cpu().numpy().view(np.uint64).tolist() == ref["counters"].tolist(), "totalReads / ignoredReads differ"
            checked += ["sum_as", "n_hit", "first_idx", "totalReads", "ignoredReads"]
        pipe._clean = False
        mine = {c: (s_, h_, n_) for sp in out for (c, s_, h_, n_) in out[sp]}
        want = {c: (s_, h_, n_) for sp in ref["result"] for (c, s_, h_, n_) in ref["result"][sp]}
        if world == 1:
            assert out == ref["result"], "chosen alleles / consensus / holes / SNPs (or their dict order) differ from the C port on the full workload"
            checked += ["species and locus order", "chosen alleles", "consensus", "holes", "snps"]
        else:
            assert all(mine.get(c) == v for c, v in want.items()), "this rank's loci differ from the C port on the full workload"
            checked += ["chosen alleles", "consensus", "holes", "snps (this rank's loci inside the merged result)"]
        ok = torch.tensor([1], dtype=torch.int32, device=device)
        if world > 1:
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
        line["parity_full_workload"] = {"ok": bool(ok.item()), "against": "oracle/c via oracle/cpu_path.py (C port of the oracle), same records", "records": w.n,
                                        "chosen_contig_records": ref["chosen_contig_records"], "piled_records": ref["piled_records"], "checked": checked,
                                        "ranks": world}
        if rank == 0 and world == 1:
            line["cpu_baseline"] = {"value": rate, "unit": "records/s", "cores": ncpu, "kind": "port", "sample": sample, "seconds_by_phase": phases,
                                    "host_cpus": os.cpu_count()}
            if not args.no_extras:
                r1, dt1, _r, sample1, ph1 = cpu_port_run(w, args, 1, steps=1)
                line["cpu_baseline"]["single_thread"] = {"value": r1, "unit": "records/s", "cores": 1, "seconds_by_phase": ph1}
        del w
    if world > 1 and not args.no_extras:
        # the other exchange form on the same shards, and the row-sharded Hamming sweep (configs[4])
        line["other_exchange"] = []
        for other in [x for x in ("p2p", "gather", "allreduce") if x != args.exchange]:
            pipe2 = pipeline.DevicePipeline(st, index, db.row_seq, impl=args.pileup_impl, idx_base=rank * R_local, exchange=other, **PARAMS)
            for _ in range(3):
                res2 = pipe2.step()
            assert res2 == result, "the exchange forms disagree"
            pipe2.capture()
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(args.steps):
                pipe2.enqueue_step()
            f1.record()
            barrier()
            assert pipe2.collect() == result
            t2 = torch.tensor([f0.elapsed_time(f1) / args.steps], dtype=torch.float64, device=device)
            torch.distributed.all_reduce(t2, op=torch.distributed.ReduceOp.MAX)
            line["other_exchange"].append({"exchange": other, "schedule": "serial passes on one stream", "ms_per_step": float(t2.item()),
                                           "value": R_total / (float(t2.item()) / 1e3), "unit": "records/s"})
            del pipe2
        line["hamming_sharded"] = extra_hamming(device, peak, world=world, rank=rank)
    if rank == 0 and world == 1 and not args.no_extras:
        line["uncapped"] = extra_uncapped(db, args, device, index, peak)
        line["hamming"] = extra_hamming(device, peak)
        line["coverage_column"] = extra_coverage(db, args, device, index)
        if args.ingest_reads:
            line["ingest"] = extra_ingest(db, args, device)
    if rank == 0:
        hs = line.get("hamming_sharded") or line.get("hamming")
        if hs:  # LAST key of the line on purpose: the driver keeps the tail of the output
            line["hamming_scaling"] = {"n": world, "all_pairs_ms": hs["all_pairs"]["ms"], "all_pairs_tensor_core_ms": hs.get("all_pairs_tensor_core", {}).get("ms"),
                                       "locus_restricted_ms": hs["locus_restricted"]["ms"], "matvec_ms": hs["matvec_one_query_per_locus"]["ms"]}
        emit(line)
    if world > 1:
        # no destroy_process_group(): tearing a communicator down while CUDA graphs that captured its kernels are alive
        # can block forever; every rank has finished its work, so leave together and let the process exit
        torch.cuda.synchronize()
        torch.distributed.barrier()
        sys.stderr.flush()
        os._exit(0)


def extra_uncapped(db, args, device, index, peak):
    """Same sample with the htslib depth cap disabled: the full histogram work (SURVEY.md 8 H1 'uncapped mode')."""
    import torch
    from metamlst_b200 import pipeline
    st, _ = gen_streams(db, args, device, None)
    out = {}
    for impl, name in ((2, "bitsliced"), (1, "atomic")):
        pipe = pipeline.DevicePipeline(st, index, db.row_seq, impl=impl, **PARAMS)
        for _ in range(2):
            res = pipe.step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 5 if impl == 2 else 2
        for _ in range(n):
            res2 = pipe.step()
        e1.record()
        torch.cuda.synchronize()
        assert res2 == res
        out.setdefault("_res", res)
        assert res == out["_res"], "atomic and bit-sliced pileup disagree"
        tids = [index.name_to_tid[c] for sp in res for (c, _s, _h, _n) in res[sp]]
        pb, precs = pileup_alg_bytes(st, tids, args.read_len)
        pms = pipe.time_kernels(10 if impl == 2 else 2)["pileup"]
        out[name] = {"ms_per_step": e0.elapsed_time(e1) / n, "value": int(st.tid.shape[0]) / (e0.elapsed_time(e1) / n / 1e3), "unit": "records/s",
                     "pileup_ms": pms, "pileup_records": precs, "algorithmic_bytes": pb,
                     "roofline": {"bound": "hbm", "achieved": pb / pms / 1e6, "peak": peak, "unit": "GB/s", "frac": pb / pms / 1e6 / peak,
                                  "traffic": ncu_traffic("pileup_uncapped_" + name) if args.reads == 10_000_000 and args.k == 4 else None},
                     "increments_per_s": precs * args.read_len * 0.94 / (pms / 1e3)}
        del pipe
    del out["_res"]
    del st
    torch.cuda.empty_cache()
    return out


def extra_ingest(db, args, device):
    """From a BAM FILE to the result (SURVEY.md 8f rank 1): the bytes of a bowtie2-ordered (name-grouped, unsorted) BAM of this workload's
    shape sit in page-locked host memory; `bam.ingest_bam` ships the COMPRESSED bytes, inflates the BGZF blocks with the hardware
    decompression engine, chains / parses / sorts / depth-caps / packs the records in HBM (csrc/ingest.cu).  Timed: host wall clock around the
    synchronous call (H2D inside), 3 repetitions; per-phase device times from CUDA events.  Parity: every array of both streams equals the
    C++ host unpacker's (mmlst_bam_unpack, all host threads, timed beside it on the same file)."""
    import tempfile
    import torch
    from metamlst_b200 import api, bam, packing, pipeline, synth
    out = {}
    for order, reps in (("name", 3), ("coord", 2)):
        cores = gen_cores(db, args, device, None, seed=1002, n_reads=args.ingest_reads)
        raw = synth.write_bam_fast(db, cores, order=order, align_records=True)
        del cores
        torch.cuda.empty_cache()
        pinned = torch.from_numpy(raw.copy()).pin_memory()
        st = bam.ingest_bam(pinned, device)          # warm-up (driver entry points, allocator)
        n = int(st.tid.shape[0])
        del st
        torch.cuda.synchronize()
        times, phases = [], None
        for _ in range(reps):
            t0 = time.perf_counter()
            st = bam.ingest_bam(pinned, device)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
            phases = st.ingest_seconds
            stats = st.ingest_stats
            if _ + 1 < reps:
                del st
        dt = min(times)
        # BAM bytes -> typed sample: ingest + one pass of the device pipeline
        index = api.AlleleIndex(st.ref_names)
        t0 = time.perf_counter()
        st2 = bam.ingest_bam(pinned, device)
        pipe = pipeline.DevicePipeline(st2, index, db.row_seq, impl=args.pileup_impl, **PARAMS)
        t1 = time.perf_counter()
        res = pipe.step()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        del pipe, st2
        # parity + host baseline: the C++ unpacker on the same file
        with tempfile.NamedTemporaryFile(suffix=".bam", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as fh:
            fh.write(raw.tobytes()); fh.flush()
            t0h = time.perf_counter()
            soa = bam.unpack_bam(fh.name, pinned=False, threads=os.cpu_count() or 1)
            t_host = time.perf_counter() - t0h
        h = lambda t: t.cpu().numpy()
        same = (np.array_equal(h(st.tid).view(np.uint32), soa.tid) and np.array_equal(h(st.as0), soa.as0) and np.array_equal(h(st.xm3), soa.xm3) and
                np.array_equal(h(st.qlen).view(np.uint16), soa.qlen) and (soa.orig_idx is None or np.array_equal(h(st.orig_idx).view(np.uint32), soa.orig_idx)) and
                np.array_equal(h(st.p_recs).reshape(-1).view(packing.PREC_DTYPE), soa.p_recs) and np.array_equal(h(st.planes).view(np.uint32), soa.planes) and
                np.array_equal(st.contig_start, soa.contig_start) and np.array_equal(h(st.qhash).view(np.uint64), soa.qhash))
        assert same, "device ingest differs from the host unpacker"
        out[order] = {"records": n, "bam_bytes": int(raw.size), "inflated_bytes": stats["inflated_bytes"], "bgzf_blocks": stats["bgzf_blocks"],
                      "seconds": dt, "seconds_all_reps": times, "records_per_s": n / dt, "bam_GBps": raw.size / dt / 1e9, "inflated_GBps": stats["inflated_bytes"] / dt / 1e9,
                      "device_seconds_by_phase": phases, "device_seconds_total": float(sum(phases.values())), "boundary_repairs": stats["boundary_repairs"],
                      "bam_to_result_seconds": t2 - t0, "of_which_pipeline_pass": t2 - t1, "loci_typed": sum(len(v) for v in res.values()),
                      "host_unpacker": {"seconds": t_host, "records_per_s": n / t_host, "threads": os.cpu_count(), "phases": soa.unpack_seconds},
                      "speedup_vs_host_unpacker": t_host / dt, "parity": "every array of both streams equals the host unpacker's",
                      "order": "bowtie2 output order (name-grouped; the device sorts)" if order == "name" else "coordinate-sorted (--presorted: no sort)"}
        del st, soa, pinned
        torch.cuda.empty_cache()
    return out


def extra_coverage(db, args, device, index):
    """Coverage column (H7): unique-QNAME dedupe of the whole score stream (hash set in HBM, 128-bit CAS).  Off the headline
    pass: display-only in the reference (metamlst.py:230), so it is timed on its own."""
    import torch
    from metamlst_b200 import pipeline
    st, _ = gen_streams(db, args, device, args.max_depth or None, want_qhash=True)
    pipe = pipeline.DevicePipeline(st, index, db.row_seq, impl=args.pileup_impl, **PARAMS)
    cov = pipe.run_coverage()
    ts = []
    for _ in range(5):
        cov2, t = pipe.run_coverage(timed=True)
        assert cov2 == cov
        ts.append(t)
    R = int(st.tid.shape[0])
    k = float(np.median([t["kernels_ms"] for t in ts])); m = float(np.median([t["memset_ms"] for t in ts]))
    out = {"kernels_ms": k, "table_memset_ms": m, "records_per_s": R / ((k + m) / 1e3), "table_bytes": ts[0]["table_bytes"],
           "stream_bytes": 25 * R, "loci": len(cov), "bases_total": int(sum(cov.values())),
           "bound": "random 32-byte sector access (hash set), not streaming"}
    del pipe, st
    torch.cuda.empty_cache()
    return out


def extra_hamming(device, peak, n_rows=1_000_000, n_q=10_000, world=1, rank=0):
    """configs[4]: 10 k reconstructed loci vs 1 M DB alleles (length 480 +- 60), all-pairs and locus-restricted.
    world > 1: the DB rows are sharded over the ranks (queries replicated), best[q] = (distance << 32 | global row) is
    all-reduced with MIN inside the timed region (strong scaling: the same 10 k x 1 M sweep on N GPUs)."""
    import torch
    from metamlst_b200 import devpack, dist, native
    g = torch.Generator(device=device); g.manual_seed(1005)
    W = 24
    lens = (480 + torch.randint(-60, 61, (n_rows,), generator=g, device=device)).to(torch.int64)
    n_loci = 1000
    hi = torch.zeros((n_rows, W), dtype=torch.int32, device=device)
    lo = torch.zeros((n_rows, W), dtype=torch.int32, device=device)
    base = torch.randint(0, 4, (n_loci, W * 32), generator=g, device=device, dtype=torch.uint8)
    per = n_rows // n_loci
    col = torch.arange(W * 32, device=device)[None, :]
    for c0 in range(0, n_rows, 100_000):
        c1 = min(n_rows, c0 + 100_000)
        codes = base[(torch.arange(c0, c1, device=device) // per).clamp(max=n_loci - 1)].clone()
        mut = torch.rand(codes.shape, generator=g, device=device) < (5.0 / 480)
        codes = torch.where(mut, (codes + torch.randint(1, 4, codes.shape, generator=g, device=device, dtype=torch.uint8)) % 4, codes)
        valid = col < lens[c0:c1, None]
        hi[c0:c1] = devpack._pack_words(((codes & 2) != 0) & valid)
        lo[c0:c1] = devpack._pack_words(((codes & 1) != 0) & valid)
    qsrc = torch.randint(0, n_rows, (n_q,), generator=g, device=device)
    qsrc = torch.sort(qsrc).values
    q_hi, q_lo, q_len = hi[qsrc].contiguous(), lo[qsrc].contiguous(), lens[qsrc].to(torch.int16)
    flip = torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32) & torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32) \
        & torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32) & torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32) \
        & torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32) & torch.randint(0, 2 ** 31 - 1, (n_q, W), generator=g, device=device, dtype=torch.int32)
    qvalid = devpack._pack_words(col < lens[qsrc][:, None])
    q_hi = (q_hi ^ (flip & qvalid)).contiguous()  # ~1/64 of the bases substituted
    def tile(x):
        nt = (x.shape[0] + 31) // 32
        p = torch.zeros((nt * 32, W), dtype=torch.int32, device=device)
        p[:x.shape[0]] = x
        return p.view(nt, 32, W).transpose(1, 2).contiguous().view(-1)
    shard = dist.shard_rows(n_rows, world, rank) if world > 1 else (0, n_rows)
    # N > 1: the all-pairs sweep (milliseconds) is sharded by DB rows and its best[] all-reduced with MIN (strong scaling); the two searches that
    # take tens of microseconds on ONE GPU are left whole on every rank (replicas): a collective costs more than the kernel (r1: 42 -> 73 us at N=8)
    db_sharded = (tile(hi[shard[0]:shard[1]]), tile(lo[shard[0]:shard[1]]), lens[shard[0]:shard[1]].to(torch.int16).contiguous())
    db_whole = db_sharded if world == 1 else (tile(hi), tile(lo), lens.to(torch.int16).contiguous())
    best = torch.empty(n_q, dtype=torch.int64, device=device)
    lib = native.lib()
    stream = torch.cuda.current_stream().cuda_stream
    out = {}
    # locus-restricted blocks: queries are sorted by source row => by locus
    qloc = (qsrc // per).clamp(max=n_loci - 1).cpu().numpy()
    blocks = []
    i = 0
    while i < n_q:
        j = i
        while j < n_q and qloc[j] == qloc[i]:
            j += 1
        l = int(qloc[i])
        blocks.append((i, j, l * per, n_rows if l == n_loci - 1 else (l + 1) * per))
        i = j
    # mat-vec regime (what a real metamlst-merge call looks like, SURVEY.md 8d): ONE query per locus => every DB row is
    # used once, the kernel streams the DB: the first query of every locus-restricted block
    mv = [(b[0], b[0] + 1, b[2], b[3]) for b in blocks]
    modes = {"all_pairs": (np.asarray([[0, n_q, 0, n_rows]], np.uint32), n_rows, n_q),
             "locus_restricted": (np.asarray(blocks, np.uint32), max(b[3] - b[2] for b in blocks), max(b[1] - b[0] for b in blocks)),
             "matvec_one_query_per_locus": (np.asarray(mv, np.uint32), max(b[3] - b[2] for b in mv), 1)}
    S = 2 * W * 4
    lens_h = lens.cpu().numpy()
    qlen_h = lens_h[qsrc.cpu().numpy()]
    popc_peak = 148 * 16 * 1.965e9  # POPC: 16 lanes/clk/SM on the XU pipe (B300_MICROARCH int table; ncu: XU 54-72 % busy)

    def alg_words(blk):
        """sum over compared pairs of ceil(min(len_q, len_r) / 32): the 32-base words stringDiff's zip really covers."""
        tot = 0
        for q0, q1, r0, r1 in blk.tolist():
            hq = np.bincount(-(-qlen_h[q0:q1] // 32), minlength=W + 1).astype(np.float64)
            hr = np.bincount(-(-lens_h[r0:r1] // 32), minlength=W + 1).astype(np.float64)
            m = np.minimum.outer(np.arange(W + 1), np.arange(W + 1))
            tot += float(hq @ m @ hr)
        return tot

    for name, (blk, mr, mq) in modes.items():
        sharded = world > 1 and name == "all_pairs"
        (sh0, sh1), (db_hi, db_lo, row_len) = (shard, db_sharded) if sharded else ((0, n_rows), db_whole)
        n_loc = sh1 - sh0
        # this rank's part of every block: rows clipped to [sh0, sh1) and rebased; blocks without local rows are dropped
        loc = blk.astype(np.int64).copy()
        loc[:, 2] = np.clip(loc[:, 2], sh0, sh1) - sh0
        loc[:, 3] = np.clip(loc[:, 3], sh0, sh1) - sh0
        loc = loc[loc[:, 3] > loc[:, 2]]
        if loc.shape[0] == 0:
            loc = np.asarray([[0, 0, 0, 0]], np.int64)
        mr = int((loc[:, 3] - loc[:, 2]).max())
        blk_d = torch.from_numpy(loc.astype(np.uint32).view(np.int32).reshape(-1)).to(device)
        def run():
            best.fill_(-1)
            native.check(lib.mmlst_hamming_min_dev2(native.ptr(db_hi), native.ptr(db_lo), native.ptr(row_len), n_loc, W, native.ptr(q_hi), native.ptr(q_lo),
                                                    native.ptr(q_len), n_q, native.ptr(blk_d), int(loc.shape[0]), max(mr, 1), int(mq), sh0, native.ptr(best), stream))
            if sharded:
                dist.allreduce_best(best)
        run(); run()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3 if name == "all_pairs" else 20
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        if world > 1:
            tm = torch.tensor([ms], dtype=torch.float64, device=device)
            torch.distributed.all_reduce(tm, op=torch.distributed.ReduceOp.MAX)
            ms = float(tm.item())
        pairs = float(sum((int(b[1]) - int(b[0])) * (int(b[3]) - int(b[2])) for b in blk))
        nq_used = int(sum(int(b[1]) - int(b[0]) for b in blk))
        comp = n_rows * S + nq_used * S + 8 * nq_used
        words = alg_words(blk)
        res = best.cpu().numpy().view(np.uint64)
        found = res != np.uint64(0xFFFFFFFFFFFFFFFF)
        qpr = pairs / n_rows
        out[name] = {"ms": ms, "pairs": pairs, "pairs_per_s": pairs / (ms / 1e3), "queries_per_row": qpr,
                     "regime": "HBM-bound (mat-vec)" if qpr <= 3 else "INT/POPC-bound",
                     "compulsory_bytes": comp, "compulsory_GBps": comp / ms / 1e6, "hbm_frac": comp / ms / 1e6 / peak,
                     "algorithmic_words": words, "word_ops_per_s": words / (ms / 1e3), "popc_roof_words_per_s": popc_peak,
                     "popc_frac": words / (ms / 1e3) / popc_peak,
                     "effective_GBps_labelled_effective": pairs * S / ms / 1e6,
                     "mean_min_dist": float((res[found] >> np.uint64(32)).astype(np.float64).mean()),
                     "checksum_best": int(np.bitwise_xor.reduce(res[found] * np.uint64(0x9E3779B97F4A7C15))) if found.any() else 0}
        if name == "all_pairs":
            # the same sweep on the tensor cores (csrc/hamming_tc.cu): DB rows expanded ONCE into the e4m3 tile image (resident, like the
            # planes), queries expanded inside the timed region; best[] must be bit-identical to the POPC kernel's
            dimg = torch.empty(int(lib.mmlst_hamming_tc_image_bytes(n_loc, W, 256)), dtype=torch.uint8, device=device)
            dmax = torch.zeros((n_loc + 255) // 256, dtype=torch.int32, device=device)
            qimg = torch.empty(int(lib.mmlst_hamming_tc_image_bytes(n_q, W, 128)), dtype=torch.uint8, device=device)
            qmax = torch.zeros((n_q + 127) // 128, dtype=torch.int32, device=device)
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            native.check(lib.mmlst_hamming_tc_expand_dev(native.ptr(db_hi), native.ptr(db_lo), native.ptr(row_len), n_loc, W, 1, 256, native.ptr(dimg), native.ptr(dmax), stream))
            f1.record()
            best_tc = torch.empty(n_q, dtype=torch.int64, device=device)

            def run_tc():
                best_tc.fill_(-1)
                native.check(lib.mmlst_hamming_tc_expand_dev(native.ptr(q_hi), native.ptr(q_lo), native.ptr(q_len), n_q, W, 0, 128, native.ptr(qimg), native.ptr(qmax), stream))
                native.check(lib.mmlst_hamming_tc_search_dev(native.ptr(qimg), native.ptr(qmax), native.ptr(q_len), n_q, native.ptr(dimg), native.ptr(dmax),
                                                             native.ptr(row_len), n_loc, W, sh0, native.ptr(best_tc), stream))
                if sharded:
                    dist.allreduce_best(best_tc)
            run_tc(); run_tc()
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            assert torch.equal(best_tc, best), "tensor-core sweep differs from the POPC kernel"
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(3):
                run_tc()
            g1.record()
            torch.cuda.synchronize()
            tms = g0.elapsed_time(g1) / 3
            if world > 1:
                tm = torch.tensor([tms], dtype=torch.float64, device=device)
                torch.distributed.all_reduce(tm, op=torch.distributed.ReduceOp.MAX)
                tms = float(tm.item())
            # flops the kernel really issues: per (query tile, row tile) pair 2 * 128 * 256 * 128 per K-block, K-blocks = 3 planes x the 128-base
            # blocks the pair can reach (min of the two tiles' longest clean sequences)
            qm, dm = qmax.cpu().numpy().astype(np.int64), dmax.cpu().numpy().astype(np.int64)
            kb_pairs = 3.0 * float(np.ceil(np.minimum.outer(qm, dm) / 128.0).clip(max=W // 4).sum())
            flops = 2.0 * 128 * 256 * 128 * kb_pairs
            bf16_peak = 1613.0
            try:
                bf16_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
            except Exception:  # noqa: BLE001
                pass
            out["all_pairs_tensor_core"] = {"ms": tms, "pairs": pairs, "pairs_per_s": pairs / (tms / 1e3), "speedup_vs_popc_kernel": ms / tms,
                                            "identical_best": True, "checksum_best": out[name]["checksum_best"],
                                            "issued_flops": flops, "dense_flops_full_K": 2.0 * pairs * 3 * 32 * W, "TFLOPs": flops / (tms / 1e3) / 1e12,
                                            "roofline": {"bound": "tensor", "achieved": flops / (tms / 1e3) / 1e12, "peak": 2 * bf16_peak, "unit": "TFLOP/s",
                                                         "frac": flops / (tms / 1e3) / 1e12 / (2 * bf16_peak), "traffic": None,
                                                         "peak_source": "2 x the measured dense bf16 rate of MEASURED_PEAKS.json (8-bit operands run at twice the 16-bit rate)"},
                                            "db_image_bytes": int(dimg.numel()), "db_expand_ms_once": f0.elapsed_time(f1), "query_image_bytes": int(qimg.numel()),
                                            "how": "tcgen05.mma cta_group::1 kind::f8f6f4 (e4m3 signs, FP32 accumulate in TMEM), M=128 N=256 K=32, TMA bulk copies into a "
                                                   "4-stage ring, persistent CTA per SM; query expansion inside the timed region, DB image resident; K loop stops at the "
                                                   "last 128-base block a tile pair can reach"}
            del dimg, qimg
        if world > 1:
            out[name]["n_gpus"] = world
            out[name]["scaling"] = ("strong (rows sharded, queries replicated, all-reduce MIN of best[] inside the timed region)" if sharded else
                                    "replicas (every rank searches the whole DB: the kernel is shorter than a collective)")
    return out


if __name__ == "__main__":
    main()
