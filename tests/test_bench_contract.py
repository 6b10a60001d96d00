"""bench.py's reference arm runs without a GPU: check the output contract on it (exactly one JSON line on
stdout, the keys the driver reads) and that the product arm refuses to run without a GPU instead of
falling back to anything on the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line(bb):
    r = run_bench("--impl", "reference", "--workload", "c1-640x480", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "lens-warp Mpixels/s" and d["unit"] == "Mpixels/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["config"]["workload"] == "c1-640x480"


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_steps_are_honoured(bb, cuda_device, tmp_path):
    """--dump-outputs: the sampled output of the last timed step is float data under 64 MB and the same from run
    to run (seeded inputs); --steps sets how many launches are timed"""
    import numpy as np

    dumps, per_step = [], set()
    for steps in (2, 5):
        d = tmp_path / f"steps{steps}"
        r = run_bench("--workload", "c1-640x480", "--steps", str(steps), "--warmup", "1", "--no-secondary", "--no-cpu-baseline",
                      "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
        assert line["steps"] == steps and line["gpu_launches"] % steps == 0
        per_step.add(line["gpu_launches"] // steps)
        files = sorted(os.listdir(d))
        assert files == ["out.npy", "out_index.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        dumps.append({f: np.load(d / f) for f in files})
    assert len(per_step) == 1 and per_step.pop() >= 1
    for f in dumps[0]:
        assert dumps[0][f].dtype in (np.float32, np.float64) and dumps[0][f].size > 0
        assert np.array_equal(dumps[0][f], dumps[1][f]), f


def test_product_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = run_bench("--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
