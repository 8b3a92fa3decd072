"""bench.py's command-line contract on the host: the reference arm (`--impl reference`, the CPU restatement timed on the host cores)
prints exactly ONE JSON line on stdout with the keys the driver reads, rank > 0 prints nothing, and the product arm refuses to run
without a GPU instead of falling back.  A short clip and a handful of tokens keep this to seconds; the real sizes run on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

try:
    import torch
    HAS_GPU = torch.cuda.is_available()
except Exception:  # pragma: no cover
    HAS_GPU = False


def _run(extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1", "--clip-seconds", "2", "--max-tokens", "4"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"].startswith("RTFx") and d["unit"] == "audio-seconds/second"
    assert d["steps"] == 1 and d["n_gpus"] == 1 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and abs(d["value"] - 2.0 / (d["ms_per_step"] / 1000.0)) < 1e-6 * d["value"] + 1e-9
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_rank0_only():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--clip-seconds", "2", "--max-tokens", "4"],
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(HAS_GPU, reason="checks the no-GPU failure mode")
def test_product_arm_has_no_cpu_fallback():
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and r.stdout.strip() == "" and "no CPU fallback" in r.stderr


def test_steps_and_dump_arguments_are_checked():
    r = _run(["--steps", "0"])
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    r = _run(["--impl", "reference", "--dump-outputs", "unused"])
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    r = _run(["--clips-per-gpu", "1025", "--max-tokens", "16384", "--dump-outputs", "unused"])
    assert r.returncode == 2 and "exceed 64 MB" in r.stderr
    assert not os.path.exists(os.path.join(ROOT, "unused"))


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_ids(tmp_path):
    """--dump-outputs writes the ids of the last timed step, [clips, max_tokens] in float32, the same in every run."""
    args = ["--gpus", "1", "--steps", "2", "--warmup", "1", "--clips-per-gpu", "3", "--clip-seconds", "2", "--max-tokens", "6",
            "--no-cpu-baseline", "--no-profile", "--no-pipelined", "--no-extras"]
    dumps = []
    for run in ("a", "b"):
        r = _run(args + ["--dump-outputs", str(tmp_path / run)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 2
        assert os.listdir(tmp_path / run) == ["ids.npy"]
        dumps.append(np.load(tmp_path / run / "ids.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (3, 6)
    assert (dumps[0] == np.round(dumps[0])).all() and dumps[0].min() >= 0
    assert np.array_equal(dumps[0], dumps[1])
