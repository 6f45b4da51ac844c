"""bench.py's reference arm runs on the host alone, so its JSON line -- the contract the driver parses -- is checked here:
one line on stdout, the required keys, a `config` that names the sample actually run, ranks other than 0 silent."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT

REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
            "data", "config", "cpu_baseline", "e2e"}


def _run(env_extra=None, args=()):
    env = dict(os.environ)
    env.update(env_extra or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--alleles", "16", "--reads", "2000",
                        *args], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout.decode()


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = _run()
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["unit"] == "records/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == d["value"] and "records" in cb["sample"]
    assert d["config"]["workload"].startswith("configs[1]") and "2000 x 150 bp" in d["config"]["workload"]  # the sample actually run
    assert "WHOLE sample" in cb["sample"] and set(d["seconds_by_phase"]) >= {"score", "select", "depthcap_pileup_consensus"}


def test_reference_arm_other_ranks_exit_silently():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}).strip() == ""


DUMPED = ("allele", "consensus_len", "consensus", "holes", "snps", "reads")


def _load_dump(d):
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in DUMPED)
    out = {n: np.load(os.path.join(d, n + ".npy")) for n in DUMPED}
    assert all(a.dtype == np.float64 and a.ndim == 1 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def test_dump_outputs_is_deterministic_and_self_consistent(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    _run(args=("--dump-outputs", str(a)))
    _run(args=("--steps", "2", "--dump-outputs", str(b)))
    da, db = _load_dump(a), _load_dump(b)
    for n in DUMPED:
        assert np.array_equal(da[n], db[n]), n
    n_loci = len(da["allele"])
    assert n_loci > 0 and len(da["holes"]) == len(da["snps"]) == len(da["consensus_len"]) == n_loci
    assert da["consensus_len"].sum() == len(da["consensus"]) and set(np.unique(da["consensus"]).tolist()) <= set(map(float, b"ACGTNacgtn"))
    assert da["reads"][0] == 2000 * 4 and 0 <= da["reads"][1] <= da["reads"][0]
