"""bench.py's reference arm runs on a CPU-only box and prints the JSON line the driver expects."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-batch", "256", "--workload", "dcn"],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    have_ref = any(os.path.isdir(os.path.join(root, "deepctr_torch"))
                   for root in (os.path.join(REPO, "baseline", "_ref"), os.environ.get("CTR_REFERENCE_ROOT", "")) if root)
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["steps"] == 1 and "workload" in line["config"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_gpu_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: on a box without CUDA the product arm exits with a message instead of computing."""
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=300, cwd=REPO)
    assert out.returncode != 0
    assert "no CUDA device" in (out.stderr + out.stdout)
