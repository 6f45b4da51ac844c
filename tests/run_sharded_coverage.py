"""Worker of tests/test_coverage_column.py::test_two_ranks_print_the_reference_coverage (launched by torch.distributed.run).

argv: bam db min_read_len out.json.  Every rank types the BAM with SampleTyper(engine="device", ingest="host") -- each scores a
contiguous range of the sorted record stream -- with the screen output on; rank 0 writes the coverage behind every allele table it
printed to out.json."""
import json
import os
import sys

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from metamlst_b200 import sample  # noqa: E402


def main():
    path, db, min_len, out = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank = torch.distributed.get_rank()
    seen = {}
    real = sample._screen_allele_table

    def spy(call, genes, coverage, longest):
        seen.update({call.species + "_" + g: int(coverage[call.species + "_" + g]) for g in genes})
        return real(call, genes, coverage, longest)
    sample._screen_allele_table = spy
    typer = sample.SampleTyper(db, device=local, engine="device", ingest="host", min_read_len=min_len)
    res = typer.type_bam(path, os.path.join(os.path.dirname(out), "rank%d" % rank), want_stdout=True)
    typer.close()
    assert res.stdout
    torch.distributed.barrier()
    if rank == 0:
        with open(out, "w") as f:
            json.dump(seen, f)
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
