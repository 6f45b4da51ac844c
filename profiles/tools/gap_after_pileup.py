import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))
import torch
sys.argv = sys.argv[:1]
import bench
from metamlst_b200 import api, native, pipeline
args = bench.parse()
dev = "cuda:0"; torch.cuda.set_device(0)
lib = native.lib()
db = bench.make_db(args)
index = api.AlleleIndex(db.ref_names())
sts = [bench.gen_streams(db, args, dev, 8000, None, seed=1002 + 100 * i)[0] for i in range(2)]
pipes = [pipeline.DevicePipeline(x, index, db.row_seq, **bench.PARAMS) for x in sts]
for p in pipes:
    for _ in range(3): p.step()
TLW = 8192
buf = torch.zeros(2 * TLW, dtype=torch.int64, device=dev)
p = pipes[0]
FL = native.SELECT_CONSUME | native.SELECT_SCRATCH_CLEAN
def seq(kind):
    p.run_score(reset=False)
    p._select_call(FL)
    p._pileup_call()
    if kind == "select": p._select_call(FL)
    elif kind == "pileup": p._pileup_call()
    elif kind == "consensus": p._consensus_call(native.CONSENSUS_CONSUME)
    elif kind == "memset": p.scratch[:64].zero_()
for kind in ("consensus", "select", "pileup"):
    native.check(lib.mmlst_debug_timeline(buf.data_ptr()))
    p.reset_tables(); seq(kind); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    p.reset_tables(); torch.cuda.synchronize()
    with torch.cuda.graph(g):
        seq(kind)
    pipes[1].step(); torch.cuda.synchronize()
    buf.zero_(); p.reset_tables(); torch.cuda.synchronize()
    g.replay(); torch.cuda.synchronize()
    native.check(lib.mmlst_debug_timeline(0))
    t = buf.cpu().numpy().astype(np.int64)[:TLW].reshape(-1, 8)
    pile_end = t[128:128 + 296, 7].max(); pile_entry = t[128:128 + 296, 0]; pile_entry_min = pile_entry[pile_entry > 0].min(); pile_entry_max = pile_entry.max()
    if kind == "consensus": nxt = t[896:896 + 21, 0].min()
    elif kind == "select": nxt = t[0:21, 0].min()
    else: nxt = None
    print(kind, "pileup entry %.2f..%.2f end(max) %.2f" % (0, (pile_entry_max - pile_entry_min) / 1e3, (pile_end - pile_entry_min) / 1e3),
          "next kernel entry +%.2f us after the last pileup CTA" % ((nxt - pile_end) / 1e3) if nxt else "second pileup: entry spread tells")
    p._clean = False
