"""Worker of tests/test_ingest_sharded.py::test_two_ranks_type_every_golden_sample (launched by torch.distributed.run): every golden
sample through SampleTyper(ingest="device", engine="device") on two ranks, each reading half of the BAM (bam.ingest_bam_sharded).
Rank 0's files and stdout must be the reference's; each rank's streams must equal its emulated shard (bam.ingest_bam_local)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from metamlst_b200 import bam, sample  # noqa: E402
from test_sample_driver import MAN, _check_against_golden, _params  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def main():
    out_root = sys.argv[1]
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
    cases = sorted(k for k in MAN if os.path.exists(os.path.join(GOLDEN, k, "sample.bam")))
    for name in cases:
        d = os.path.join(GOLDEN, name)
        path = os.path.join(d, "sample.bam")
        prm = _params(name)
        st = bam.ingest_bam_sharded(path, local, presorted=prm["presorted"])
        emu = bam.ingest_bam_local(path, world, local, presorted=prm["presorted"])[rank]
        for k in ("tid", "as0", "xm3", "qlen", "orig_idx", "qhash", "p_recs", "planes"):
            assert torch.equal(getattr(st, k), getattr(emu, k)), (name, rank, k)
        assert np.array_equal(st.contig_start, emu.contig_start) and st.n_dropped == emu.n_dropped, (name, rank)
        typer = sample.SampleTyper(os.path.join(d, "db.sqlite"), device=local, engine="device", ingest="device", **prm)
        out = os.path.join(out_root, name)
        res = typer.type_bam(path, out, want_stdout=True, timestamp=7)
        typer.close()
        torch.distributed.barrier()
        if rank == 0:
            _check_against_golden(name, res, out)
    torch.distributed.barrier()
    if rank == 0:
        print("SHARDED-INGEST-OK", len(cases))
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
