"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) prints ONE JSON line with the keys the driver
reads, and the product arm refuses to run without a CUDA device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import torch

from helpers import ROOT


def _run(*args, timeout=600):
    env = dict(os.environ, OMP_NUM_THREADS="8")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--batch", "2")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "graph-steps/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    # the reference arm describes the SAME workload object as the product arm launched with the same flags (what it samples of it is
    # said in `sample` / `cpu_baseline.sample`, never in `config`)
    sys.path.insert(0, ROOT)
    import bench
    bench.L = bench.WORKLOADS["cfg2"]["L"]
    assert d["config"] == bench.workload_config(bench.WORKLOADS["cfg2"], 2, bench.WORKLOADS["cfg2"]["T"], 1)
    assert "one denoise step" in d["sample"].lower()
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_same_arguments_same_arrays(tmp_path):
    """--dump-outputs writes the last timed step's arrays as .npy; two runs with the same arguments dump identical arrays, and
    --steps below 1 is refused rather than changed."""
    import numpy as np
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = _run("--impl", "reference", "--steps", "2", "--warmup", "0", "--batch", "2", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        dumps.append({p.name: np.load(p) for p in sorted(d.glob("*.npy"))})
    assert sorted(dumps[0]) == ["logits.npy", "x.npy"]
    for name, a in dumps[0].items():
        assert a.dtype == np.float32 and a.shape == (2, 128, 20) and np.isfinite(a).all()
        assert np.array_equal(a, dumps[1][name]), name
    assert sum(a.nbytes for a in dumps[0].values()) <= 64 << 20
    r = _run("--impl", "reference", "--steps", "0", "--warmup", "0", "--batch", "2", timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_recorded_product_and_reference_lines_share_one_config():
    """the two lines of the last B200 verification of the round (profiles/): same metric, unit, direction and config object."""
    a = json.load(open(os.path.join(ROOT, "profiles", "bench_r02_final2.json")))
    b = json.load(open(os.path.join(ROOT, "profiles", "bench_ref_r02_final2.json")))
    assert b["impl"] == "reference" and "impl" not in a
    for k in ("metric", "unit", "higher_is_better", "config"):
        assert a[k] == b[k], k
    assert a["gpu_launches"] > 0 and a["e2e"]["h2d_bytes_per_step"] > 0 and a["e2e"]["d2h_bytes_per_step"] > 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_has_no_cpu_fallback():
    if torch.cuda.is_available():
        return
    r = _run("--steps", "1", "--warmup", "0", timeout=120)
    assert r.returncode != 0
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert "error" in d and "no CPU fallback" in d["error"]
