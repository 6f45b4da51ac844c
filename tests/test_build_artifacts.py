"""What the compiler made of the hot kernels, checked without a GPU on the objects `build()` leaves in csrc/: the ring score
kernel and the bit-sliced pileup really move their tiles with TMA bulk copies completing on mbarriers (SASS `UBLKCP`, `SYNCS`),
the warp reductions are single `REDUX` instructions, the Hamming kernel counts with `POPC`, and the hot kernels do not spill
registers to local memory (ptxas -v logs; the pileup kernel is allowed the 16 bytes it parks outside its loop)."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "metamlst_b200", "csrc")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _sass(obj):
    path = os.path.join(CSRC, obj)
    if not os.path.exists(path) or not os.path.exists(CUOBJDUMP):
        pytest.skip("needs the objects of build() and cuobjdump")
    out = subprocess.run([CUOBJDUMP, "-sass", path], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=300).stdout.decode(errors="replace")
    funcs = {}
    cur = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def test_ring_score_kernels_use_tma_and_mbarriers():
    f = _sass("score_runs.o")
    ring = {k: v for k, v in f.items() if "ring" in k}
    assert len(ring) >= 9, sorted(f)
    for name, sass in ring.items():
        assert "UBLKCP" in sass, name          # cp.async.bulk: the stages are filled by the TMA unit
        assert "SYNCS" in sass, name           # mbarrier arrive.expect_tx / try_wait
        assert "REDUX" in sass, name           # warp sums as one instruction
        assert "IDP" in sass, name             # dp2a: masked sum of two int16 per instruction
        assert not re.search(r"\b(LDL|STL)\b", sass), name  # no local-memory traffic
    regs = [v for k, v in f.items() if "score_runs_kernel" in k]
    assert regs and all("UBLKCP" not in v for v in regs)  # the register forms load through LDG only


def test_pileup_and_hamming_instruction_selection():
    p = _sass("pileup_bitsliced.o")
    kern = [v for k, v in p.items() if "pileup_bitsliced_kernel" in k]
    assert kern and all("UBLKCP" in v and "SYNCS" in v and "LOP3" in v for v in kern)
    h = _sass("hamming.o")
    kern = [v for k, v in h.items() if "hamming_min_kernel" in k]
    assert kern and all("POPC" in v and "LDGSTS" in v for v in kern)  # popcount distance, cp.async query staging


def test_tensor_core_hamming_uses_tcgen05_tmem_and_tma():
    """csrc/hamming_tc.cu: `tcgen05.mma` shows as UTC*MMA, `tcgen05.ld` as LDTM, `tcgen05.commit` as UTCBAR, TMEM allocation as UTCATOMSWS,
    the stage fills as UBLKCP; nothing of the legacy tensor path (HMMA from mma.sync / wmma)."""
    f = _sass("hamming_tc.o")
    kern = [v for k, v in f.items() if "hamming_tc_kernel" in k]
    assert len(kern) == 1
    k = kern[0]
    assert re.search(r"\bUTC[A-Z]*MMA\b", k) and "LDTM" in k and "UTCBAR" in k and "UTCATOMSWS" in k and "UBLKCP" in k and "SYNCS" in k
    assert not re.search(r"\bHMMA\b", k) and not re.search(r"\b(LDL|STL)\b", k)


def test_ingest_kernels_are_built_and_do_not_spill():
    f = _sass("ingest.o")
    names = " ".join(f)
    for k in ("chain_guess_kernel", "chain_repair_kernel", "chain_offsets_kernel", "parse_kernel", "gather_kernel", "cap_kernel", "pack_kernel"):
        assert k in names, k
    pack = [v for k, v in f.items() if "pack_kernel" in k][0]
    assert "VOTE" in pack   # the plane words are assembled by warp ballots
    text = open(os.path.join(CSRC, "ingest.ptxas.log")).read()
    for m in re.finditer(r"Compiling entry function '(\S+)'.*?\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", text):
        if any(k in m.group(1) for k in ("chain_", "parse_kernel", "gather_kernel", "cap_kernel", "pack_kernel")):
            assert int(m.group(3)) == 0 and int(m.group(4)) == 0, m.group(1)


def test_hot_kernels_do_not_spill():
    bad = []
    for log in ("score_runs", "score", "pileup_bitsliced", "hamming", "select", "consensus", "coverage"):
        path = os.path.join(CSRC, log + ".ptxas.log")
        if not os.path.exists(path):
            pytest.skip("needs the ptxas logs of build()")
        text = open(path).read()
        for m in re.finditer(r"Compiling entry function '(\S+)'.*?\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", text):
            name, _stack, st, ld = m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))
            if "pileup_bitsliced" in name:
                # 128 registers at 2 CTAs per SM hold 50 bit-sliced counter planes: ptxas parks a few bytes outside the tile loop
                if st > 32 or ld > 32:
                    bad.append((name, st, ld))
            elif (st or ld) and ("ring" in name or "hamming_min" in name or "ILb0ELb0ELb1E" in name):
                bad.append((name, st, ld))
            elif "coverage_cu" in name and (_stack or st or ld):  # insert / merge / sum passes of the coverage column
                bad.append((name, _stack, st, ld))
    assert not bad, bad
