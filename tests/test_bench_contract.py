"""bench.py's contract on a GPU-less host: the reference arm prints ONE JSON line with the keys the driver reads, on the
same metric / unit / config as the GPU arm, and a non-zero rank under torchrun prints nothing and exits 0.

--dump-outputs: on the GPU, the file holds exactly what the last timed step returned; on the CPU, oversized arrays keep a
fixed sample of whole rows within the size budget, and arguments that cannot be honoured are refused."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _run(env_extra, *args):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)


def test_reference_arm_prints_one_contract_line():
    res = _run({}, "--impl", "reference", "--steps", "1", "--warmup", "0")
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout[-2000:]
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "streams_x_frames_per_sec" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "streams" in cb["sample"]
    assert cb["cores"] == cb["host"]["threads_used"] <= cb["host"]["affinity"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "configs[1]" in d["config"]["workload"] and "model" not in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    res = _run({"RANK": "3", "WORLD_SIZE": "8", "LOCAL_RANK": "3"}, "--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "0")
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_steps_below_one_and_reference_dump_are_rejected(tmp_path):
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", str(tmp_path))):
        res = _run({}, *args)
        assert res.returncode == 2 and "usage" in res.stderr, (args, res.stderr[-2000:])
    assert not any(tmp_path.iterdir())


def test_dump_outputs_keeps_a_fixed_row_sample_within_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100 * 101 * 4 + 4096)
    probs = np.random.default_rng(1).random((1000, 101), dtype=np.float32)
    small = np.arange(12, dtype=np.float64).reshape(3, 4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"probs": probs, "small": small})
    a, b = np.load(tmp_path / "a" / "probs.npy"), np.load(tmp_path / "b" / "probs.npy")
    assert a.dtype == np.float32 and a.shape[1] == 101 and 0 < a.shape[0] < 1000 and np.array_equal(a, b)
    rows = np.flatnonzero((probs[:, None, :] == a[None, :, :]).all(2).any(1))
    assert len(rows) == a.shape[0] and np.array_equal(probs[rows], a)        # whole rows, in stream order
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.astype(np.float32))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


@pytest.mark.gpu
def test_dump_outputs_is_what_the_last_timed_step_returned(tmp_path, torch_cuda):
    import bench
    from microwakeword_b200.engine import StreamEngine
    streams, warmup, steps = 2048, 2, 3
    res = _run({}, "--streams", str(streams), "--steps", str(steps), "--warmup", str(warmup), "--no-e2e", "--no-cpu", "--no-extra",
               "--dump-outputs", str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    assert json.loads(res.stdout)["steps"] == steps
    got = np.load(tmp_path / "probs.npy")
    torch = torch_cuda
    audio = bench.synth_audio_device(torch, streams, bench.SAMPLES_PER_STEP, 1234, torch.device("cuda", 0))
    eng = StreamEngine(bench.model_blob("f32"), n_streams=streams, device=0)
    eng.reset()
    for _ in range(warmup + steps):                    # state carries over between calls: the dump is the last of them
        want = eng.predict_clip(audio)
    assert got.dtype == np.float32 and np.array_equal(got, want.cpu().numpy())
