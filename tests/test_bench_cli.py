"""bench.py contract pieces that run without a GPU: the reference arm (`--impl reference`) prints one JSON line with
the keys the driver reads, on the same 65 536-sample step as the GPU arm unless --batch says otherwise."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--batch", "2048"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["config"]["batch_per_step"] == 2048
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]


def test_reference_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    import numpy as np

    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "2", "--warmup", "1", "--batch", "1024",
                            "--dump-outputs", str(tmp_path / run)], cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
        assert [p.name for p in (tmp_path / run).iterdir()] == ["reference_predictions.npy"]
        dumps.append(np.load(tmp_path / run / "reference_predictions.npy"))
    assert dumps[0].shape == (1024, 1) and dumps[0].dtype == np.float32
    assert np.all((dumps[0] > 0) & (dumps[0] < 1))  # sigmoid head
    assert np.array_equal(dumps[0], dumps[1])


def test_default_reference_step_is_the_full_batch():
    src = (ROOT / "bench.py").read_text()
    assert "sample = min(args.cpu_sample or B, B)" in src  # same_config: 65 536 samples per CPU step by default
