"""Worker of tests/test_cmseq_device.py::test_two_ranks_gather_over_nccl (launched by torch.distributed.run): cmseq's BamFile sharded by
contig over two ranks (BamFile(ingest="device", group=WORLD)); `gather` of every `*_all` result must equal the single-GPU host route on
every rank, and each rank's contigs must be the kept contigs it owns."""
import os
import sys

import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from metamlst_b200 import cmseq_api  # noqa: E402
from test_cmseq_bulk import GOLD, _same  # noqa: E402
from test_cmseq_device import _golden_calls  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    group = torch.distributed.group.WORLD
    rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
    for scen in sorted(GOLD):
        path = os.path.join(GOLDEN, scen, "sample.bam")
        host = cmseq_api.BamFile(path, device=local)
        bf = cmseq_api.BamFile(path, device=local, ingest="device", group=group)
        own = cmseq_api.owner_map(host.lengths, world)
        assert list(bf.contigs) == [c for c in host.contigs if own[host._tid[c]] == rank], (scen, rank)
        for method, kw in _golden_calls(scen):
            _same(bf.gather(getattr(bf, method)(**kw)), getattr(host, method)(**kw), "%s:%s:rank %d" % (scen, method, rank))
        bf.close()
        host.close()
    torch.distributed.barrier()
    if rank == 0:
        print("CMSEQ-SHARDED-OK", len(GOLD))
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
