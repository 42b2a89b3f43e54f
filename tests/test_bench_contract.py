"""bench.py's reference arm runs without a GPU and its JSON line must carry the result keys; the GPU arm's extra keys are checked
here by name in the source.  On a GPU: the timed step count and the output dump."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "structured-layer fwd+bwd samples/sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("C5: SSS 4096->1000")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "batch 256" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_gpu_arm_emits_the_contract_keys():
    src = open(os.path.join(REPO, "bench.py")).read()
    for key in ("roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "h2d_bytes_per_step", "d2h_bytes_per_step", "traffic",
                "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "sm_max_mhz", "reasons"):
        assert key in src, key


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path, built_lib):
    """At batch 4096 the SSS workload rotates four input sets; --steps 3 must time exactly three steps, and --dump-outputs must hold
    the output and parameter gradients of the third one, as one eager step on the same seeded layer and inputs computes them."""
    import torch
    import bench
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "3", "--warmup", "1", "--quick", "--no-cpu-baseline",
                        "--global-batch", "4096", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3
    assert d["config"]["launch_mode"].startswith("CUDA graph"), d["config"]["launch_mode"]     # the dump must not cost the capture
    assert sorted(os.listdir(tmp_path)) == ["grad_flat.npy", "y.npy"]
    wl = bench.SSSWorkload()
    runner = bench.StepRunner(wl, torch.device("cuda"), 4096, seed=5000)
    assert runner.n_sets == 4
    y = runner.step(2)
    for name, ref in (("y", y), ("grad_flat", runner.layer.flat_grad())):
        got = np.load(tmp_path / (name + ".npy"))
        ref = ref.detach().cpu().numpy()
        assert got.dtype == np.float32 and got.shape == ref.shape, name
        assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max(), name
