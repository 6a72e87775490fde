"""bench.py's command line: the JSON-line contract of the reference arm, which runs on CPU (one line on stdout, the required
keys, the reference-arm keys), the arguments it refuses, and on the GPU the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line(orc):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nodes", "3000", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "alert_cells_per_sec_to_converged_cut" and d["unit"] == "cells/s"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and d["steps"] == 2
    # everything in cpu_baseline is measured on the sample; the whole-cluster figure is a labelled extrapolation on the side
    assert cb["sampled_nodes"] >= 1 and cb["apply_s"] > 0 and cb["tally_s"] > 0
    assert abs(cb["value"] - d["config"]["cells"] / (cb["apply_s"] + cb["tally_s"])) <= 0.5 * cb["value"]     # mean of 2 steps
    assert "NOT measured" in cb["extrapolated_whole_cluster"]["how"]


def test_reference_arm_runs_the_flip_flop_stream(orc):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c4", "--nodes", "3000",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.strip()][0])
    assert d["config"]["workload"].startswith("C4 3000-node") and d["value"] > 0


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--nodes", "3000"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and p.stdout.strip() == "", p.stderr[-2000:]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,nodes", [("c2", 2000), ("c4", 3000)])
def test_gpu_arm_dumps_the_outputs_of_its_last_timed_step(tmp_path, workload, nodes):
    import numpy as np
    env = dict(os.environ, RAPID_B200_NO_CLOCKS="1")
    runs = []
    for i in range(2):
        d = tmp_path / str(i)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--nodes", str(nodes), "--steps",
                            "3", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, env=env)
        assert p.returncode == 0, p.stderr[-3000:]
        assert json.loads([l for l in p.stdout.splitlines() if l.strip()][0])["steps"] == 3
        runs.append({f.name[:-4]: np.load(f) for f in d.iterdir()})
    a = runs[0]
    assert set(a) == {"decision", "cut", "receivers", "proposal_fingerprint", "proposal_len", "announced"}
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    decided, h1hi, h1lo, h2hi, h2lo, length = a["decision"][:6]
    assert decided == 1 and length == len(a["cut"]) > 0 and (np.diff(a["receivers"]) == 1).all() and len(a["receivers"]) == nodes
    holders = (a["proposal_fingerprint"] == [h1hi, h1lo, h2hi, h2lo]).all(axis=1) & (a["proposal_len"] == length)
    assert holders.any() and (a["announced"][holders] == 1).all()
    for k in a:                                  # same arguments, same inputs: the same outputs, bit for bit
        assert np.array_equal(a[k], runs[1][k]), k
