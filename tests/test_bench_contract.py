"""bench.py's command line, reference arm and JSON line format (CPU), and the output dump of the GPU arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=900, env=e)


def test_reference_arm_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "training volumes/sec" and d["unit"] == "volumes/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"], env={"RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--inference", "--dump-outputs", "x"]):
        r = _run(args)
        assert r.returncode == 2 and "error" in r.stderr, args


def test_dump_outputs_layout(tmp_path):
    """loss + one file per parameter, float32, within 64 MB; large tensors sampled at the same positions every time"""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import unetsulc_b200
    torch.manual_seed(0)
    model = unetsulc_b200.UNet3D(1, 56)
    loss = torch.tensor([4.0, 400.0])
    bench.dump_outputs(str(tmp_path / "a"), loss, model)
    bench.dump_outputs(str(tmp_path / "b"), loss, model)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(["loss.npy"] + ["param.%s.npy" % n for n, _ in model.named_parameters()])
    total = 0
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
        total += os.path.getsize(tmp_path / "a" / n)
    assert total <= 64 << 20
    assert np.array_equal(np.load(tmp_path / "a" / "loss.npy"), [4.0, 400.0])
    w = model.encoders[0].double_conv.conv1.weight
    assert np.array_equal(np.load(tmp_path / "a" / "param.encoders.0.double_conv.conv1.weight.npy"), w.detach().numpy())
    big = dict(model.named_parameters())["decoders.0.double_conv.conv1.weight"].detach().numpy().reshape(-1)
    s = np.load(tmp_path / "a" / "param.decoders.0.double_conv.conv1.weight.npy")
    assert s.shape == (bench.DUMP_SAMPLE,) and np.isin(s, big).all()


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    r = _run(["--steps", "3", "--warmup", "0", "--no-e2e", "--no-torch-gpu", "--no-cpu-baseline",
              "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3
    loss = np.load(tmp_path / "loss.npy")
    assert loss.shape == (2,) and np.all(np.isfinite(loss)) and 0 < loss[0] < 10
    assert len(os.listdir(tmp_path)) == 1 + 44


def test_traffic_comes_from_the_committed_ncu_capture():
    sys.path.insert(0, ROOT)
    import bench
    t, src = bench.load_traffic()
    assert t and t > 1e6 and src.startswith("profiles/")
