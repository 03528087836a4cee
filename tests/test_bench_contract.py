"""bench.py contract checks that run without a GPU: the reference arm's JSON line, and that the GPU arm refuses to run
(no CPU fallback) when there is no CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e,
                          timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["config"]["workload"].startswith("static-PTQ int8 SimpleConvNet forward")
    assert d["dtype"] == "u8" and d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dumps_the_logits_of_its_last_step(tmp_path, oracle_model):
    from convnet_quantization_b200 import synth
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / "logits.npy")
    assert got.dtype == np.float32 and got.shape == (64, 10)
    with torch.no_grad():
        want = oracle_model(synth.images_f32(64, seed=11)).numpy()
    assert np.array_equal(got, want)


def test_steps_must_be_positive():
    r = _run("--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_gpu_arm_dumps_the_logits_of_its_last_timed_step(tmp_path):
    """The dump is what ``engine.forward`` returns for the benchmark's seeded input, so two builds compare."""
    from convnet_quantization_b200 import synth
    from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel
    b = 512
    r = _run("--steps", "2", "--warmup", "1", "--batch", str(b), "--no-cpu-baseline", "--sustain-s", "0",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([ln for ln in r.stdout.splitlines() if ln.strip()]) == 1
    got = np.load(tmp_path / "logits.npy")
    assert got.dtype == np.float32 and got.shape == (b, 10)
    dev = torch.device("cuda", 0)
    m = StaticPTQModel(device=dev)
    m.fp32_model.load_state_dict(synth.make_state_dict(0))
    engine = m.quantize().engine
    g = torch.Generator(device=dev).manual_seed(0)
    x = synth.normalize(torch.randint(0, 256, (b, 3, 32, 32), dtype=torch.uint8, device=dev, generator=g)).contiguous()
    assert np.array_equal(got, engine.forward(x).cpu().numpy())


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful without a GPU")
def test_gpu_arm_has_no_cpu_fallback():
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
