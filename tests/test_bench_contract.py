"""bench.py's reference arm runs without a GPU (it times the oracle port on the host cores): check the JSON line it
prints.  On a device, the GPU arm's step count and the output it dumps are checked too."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "g1_msm_mops_2^20" and d["unit"] == "Mop/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_gpu_arm_fails_loudly_without_cuda():
    """No CPU fallback: without a device the GPU arm must exit non-zero, not print a number."""
    try:
        import torch
        if torch.cuda.is_available():
            return
    except Exception:
        pass
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-secondary"],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode != 0
    assert not any(l.strip().startswith("{") and '"value"' in l for l in out.stdout.splitlines())


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    """--steps sets the number of timed steps and --dump-outputs writes what the last of them returned: with bases b_i * G
    and the scalar set of that step, the 96 bytes are the encoding of (sum s_i b_i) * G."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--log-n", "12", "--no-cpu",
                          "--no-secondary", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == 2
    got = np.load(tmp_path / "g1_msm.npy")
    assert got.dtype == np.float64 and got.shape == (96,)
    sys.path.insert(0, ROOT)
    import bench
    from zero_chain_b200 import synthetic as sy
    n = 1 << 12
    last = bench.make_scalars(n, 0, (d["warmup"] + d["steps"] - 1) % bench.N_SETS)
    assert bytes(got.astype(np.uint8)) == bench.closed_form_g1(bench.dot_mod_r(last, sy.random_fr_limbs(n, 7)))
