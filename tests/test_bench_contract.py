"""bench.py on a machine without a GPU: the reference arm must print the contract's JSON line, and the product arm must
refuse to run (there is no CPU fallback to measure).  On the GPU: what --dump-outputs writes."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _run(*args):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 1 and line["higher_is_better"] is True
    assert line["unit"] == "Mpx/s" and line["value"] > 0 and line["ms_per_step"] > 0 and line["dtype"] == "u8"
    assert line["steps"] == 1 and line["warmup"] >= 1 and line["scaling"] == "weak" and line["data"] == "synthetic"
    assert "Mpixels/s 8K equirect->cubemap bicubic" in line["metric"] and line["config"]["workload"].startswith("cfg2")
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


@pytest.mark.gpu
def test_dumped_outputs_are_the_last_timed_step(golden, tmp_path):
    """--dump-outputs with one timed step: that step transforms frame 0 of the ring, whose luma plane the reference's
    recorded output pins; chroma planes whole, float32, within 64 MB."""
    import numpy as np
    from oracle import ref_harness as rh
    r = _run("--steps", "1", "--warmup", "3", "--skip-e2e", "--skip-cpu-baseline", "--skip-other-configs", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 1
    out = {p: np.load(tmp_path / f"out_{p}.npy") for p in "yuv"}
    assert [out[p].shape for p in "yuv"] == [(2560, 3840), (1280, 1920), (1280, 1920)]
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum((tmp_path / f"out_{p}.npy").stat().st_size for p in "yuv") <= 64_000_000
    assert rh.sha16(out["y"].astype(np.uint8)) == golden["full"]["cfg2"]["planes"]["0"]["out_sha"]


def test_product_arm_refuses_to_run_without_a_gpu():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the product arm is exercised by the gpu-marked tests and the bench itself")
    r = _run("--steps", "1")
    assert r.returncode != 0
    assert "no CUDA device" in (r.stdout + r.stderr)
