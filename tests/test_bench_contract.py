"""bench.py contract on a CPU-only box: the reference arm (the reference's algorithm on the host cores — the oracle
port, the one other place bench.py may execute oracle/) prints the JSON line the driver parses; the product arm has no CPU
fallback and fails loudly without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_line():
    p = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "rays/sec" and line["unit"] == "rays/s"
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert "configs[1]" in line["config"]["workload"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "rays" in cb["sample"]
    e = line["e2e"]
    assert e["value"] == line["value"] and e["unit"] == line["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def _dumped(d, R):
    shapes = {"rgb_values": (R, 3), "fg_rgb_values": (R, 3), "normal_values": (R, 3), "acc_map": (R,),
              "acc_person_list": (R, 2)}
    assert sorted(os.listdir(d)) == sorted(k + ".npy" for k in shapes)
    out = {k: np.load(os.path.join(d, k + ".npy")) for k in shapes}
    for k, a in out.items():
        assert a.dtype == np.float32 and a.shape == shapes[k] and np.isfinite(a).all(), k
    return out


def test_reference_arm_dump_outputs(tmp_path):
    p = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out")])
    assert p.returncode == 0, p.stderr[-2000:]
    _dumped(tmp_path / "out", 128)


@pytest.mark.gpu
def test_product_arm_dump_outputs_repeat(tmp_path):
    """Same arguments, same inputs: two runs of the timed path dump the same pixels."""
    args = ["--steps", "2", "--warmup", "0", "--no-extras", "--no-cpu-baseline", "--dump-outputs"]
    runs = []
    for i in range(2):
        d = str(tmp_path / ("run%d" % i))
        p = _run(args + [d])
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
        runs.append(_dumped(d, 4096))
    for k in runs[0]:
        assert np.array_equal(runs[0][k], runs[1][k]), k


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a box without a GPU")
def test_product_arm_has_no_cpu_fallback():
    p = _run(["--steps", "1", "--warmup", "0", "--no-extras", "--no-cpu-baseline"], timeout=300)
    out = p.stdout.strip().splitlines()
    assert p.returncode != 0
    assert not any(l.startswith("{") and '"value"' in l for l in out)
