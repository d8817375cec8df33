"""bench.py --impl reference (the reference's own CPU implementation of the path, oracle/_ref, or the oracle port
where that is not built) prints the benchmark's JSON line on a machine without a GPU; R-MAT 18 so that the whole
run ends in about half a minute."""
import json
import os
import subprocess
import sys

from oracle import bindings as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "rmat18",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().split("\n")[-1])
    assert d["impl"] == "reference" and d["metric"] == "lp_edges_per_second" and d["unit"] == "edges/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"] == "rmat18" and d["config"]["same_workload"] is True
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if B.have_parallel_reference() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "rmat18" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
