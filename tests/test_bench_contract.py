"""bench.py's reference arm runs on host cores only, so its JSON contract can be checked without a GPU; the output dump
of our arm needs one."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


ENV = dict(os.environ, PB_REF_FILL="20000")      # the driver's run fills the whole 1M-capacity buffer; keep the CPU suite short


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=600, env=ENV)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                       # ONE JSON line
    line = json.loads(lines[0])
    # --steps is the number of timed iterations; warm-ups are at least 3; "steps" / "warmup" report what was really
    # timed, the request is kept beside them
    assert line["impl"] == "reference" and line["n_gpus"] == 1 and line["steps_requested"] == 2 and line["warmup_requested"] == 1
    assert line["steps"] == 2 and line["warmup"] == 3
    assert line["cpu_baseline"]["sample"].startswith("2 hot-loop iterations after 3 warm-ups")
    assert line["unit"] == "transitions/s" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["value"] > 0 and abs(line["ms_per_step"] * 1e-3 * line["value"] - 256) < 1e-6 * 256
    assert "workload" in line["config"] and "model" not in line["config"]
    cpu = line["cpu_baseline"]
    assert cpu["kind"] in ("port", "reference") and cpu["cores"] >= 1 and cpu["value"] == line["value"] and cpu["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_under_torchrun_prints_once():
    """N > 1: launched like our own arm; rank 0 alone measures and prints, the other ranks exit 0 without work."""
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29613", os.path.join(ROOT, "bench.py"),
                          "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                         cwd=ROOT, capture_output=True, text=True, timeout=900, env=ENV)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0
    assert line["config"]["global_batch"] == 512                 # like for like with our arm at 2 GPUs (256 per GPU)


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: after exactly --steps timed steps, what the last step of each timed leg computed, as float32 /
    float64 .npy files of 64 MB at most."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--quick", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    arrays = {f[:-len(".npy")]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    for prefix in ("", "e2e_"):
        a = {k[len(prefix):]: v for k, v in arrays.items() if k.startswith(prefix)}
        assert {"loss", "td", "index", "weight", "observation", "params", "priorities"} <= set(a)
        assert np.isfinite(a["loss"]).all() and a["td"].size == 256 and a["priorities"].shape == (1_000_000,)
        assert ((a["index"] >= 0) & (a["index"] < 1_000_000)).all() and (a["index"] == np.round(a["index"])).all()
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
