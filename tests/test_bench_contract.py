"""bench.py's output contract, checked without a GPU: the reference arm (`--impl reference`: the oracle port of the
reference's CPU sweep on the host cores) prints one JSON line with the agreed keys, ranks other than 0 stay silent, and
the B200 arm refuses to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        e.pop(k, None)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-images", "16"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "calibration_images_per_s" and d["unit"] == "images/s"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["scaling"] == "strong" and d["vs_baseline"] is None and d["data"] == "synthetic"
    # the reference arm names the SAME configuration as the B200 arm (what the sample was lives in cpu_baseline.sample)
    import argparse
    import bench
    want = bench.bench_config(argparse.Namespace(model="base", sparsity=0.375, images=1024, batch=256), 1)
    assert d["config"] == want and "ViT-B/16" in d["config"]["workload"] and d["config"]["images_per_step"] == 1024
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == "images/s" and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_runs_on_rank_zero_only():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine WITHOUT a CUDA device")
def test_b200_arm_refuses_to_run_without_a_gpu():
    r = _run(["--steps", "1", "--warmup", "0"], timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())  # no number without a GPU


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step_and_repeat_exactly(tmp_path):
    """--dump-outputs saves what the timed step returned; another run on the same inputs, with another step count, saves
    the same bits; --steps sets the number of timed steps (the launches counted in the timed region scale with it)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import numpy as np
    n_img = 96
    common = ["--model", "small", "--images", str(n_img), "--batch", "32", "--warmup", "1",
              "--no-prune", "--no-extra", "--no-cpu-baseline", "--no-clocks"]
    lines, dumps = {}, {}
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        r = _run([*common, "--steps", str(steps), "--dump-outputs", str(d)], timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        lines[steps] = json.loads(next(ln for ln in r.stdout.splitlines() if ln.startswith("{")))
        dumps[steps] = {name: np.load(d / f"{name}.npy") for name in ("s1_score_sums", "ffn_importance")}
    assert lines[1]["steps"] == 1 and lines[3]["steps"] == 3
    assert lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"] > 0
    sums, imp = dumps[1]["s1_score_sums"], dumps[1]["ffn_importance"]
    assert sums.dtype == np.float32 and imp.dtype == np.float32
    assert sums.shape == (12 * 1536,) and imp.shape == (12, 1536)      # ViT-S/16: 12 blocks of 1536 neurons
    assert np.isfinite(sums).all() and (sums > 0).all()
    assert np.allclose(imp.reshape(-1), sums / n_img, rtol=1e-5)
    for name in dumps[1]:
        assert np.array_equal(dumps[1][name], dumps[3][name]), name
