"""bench.py's reference arm runs without a GPU: check the JSON contract of the line a caller parses; and the outputs
--dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                        # exactly one JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "audio samples/sec" and d["unit"] == "samples/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args),
                          capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_steps_below_one_and_reference_dump_are_refused():
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", "unused")):
        out = _bench(*args)
        assert out.returncode == 2 and "error" in out.stderr


def test_dump_outputs_keeps_dtype_and_samples_within_the_limit(tmp_path):
    import bench
    big = np.arange(100000, dtype=np.float32).reshape(10, 10000)
    limit = 3 * 4096 + 3 * 8000
    arrays = {"big": big, "f64": np.float64(1.5), "i32": np.array([3], np.int32)}
    bench.dump_outputs(str(tmp_path / "a"), arrays, limit=limit)
    bench.dump_outputs(str(tmp_path / "b"), arrays, limit=limit)
    assert sum(os.path.getsize(str(p)) for p in (tmp_path / "a").iterdir()) <= limit
    a, b = np.load(str(tmp_path / "a" / "big.npy")), np.load(str(tmp_path / "b" / "big.npy"))
    assert a.dtype == np.float32 and a.size == 2000 and np.array_equal(a, b)             # the same seeded sample
    assert np.all(np.diff(a) > 0) and np.all(np.isin(a, big))                            # elements of the output, in order
    assert np.load(str(tmp_path / "a" / "f64.npy")).dtype == np.float64
    assert np.load(str(tmp_path / "a" / "i32.npy")).dtype == np.float32


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(lib, tmp_path):
    """The student workload's dump equals a direct call on bench.py's seeded inputs; --steps sets the timed steps
    (the library's launch counter over the timed region doubles from one step to two)."""
    B, T = 2, 4096
    lines = {}
    for steps in (1, 2):
        out = _bench("--workload", "student", "--batch", str(B), "--length", str(T), "--steps", str(steps), "--warmup", "1",
                     "--dump-outputs", str(tmp_path / ("steps%d" % steps)))
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    d = lines[2]
    assert d["steps"] == 2 and d["config"]["batch_per_gpu"] == B and d["config"]["samples_per_utterance"] == T
    assert lines[1]["gpu_launches"] > 0 and d["gpu_launches"] == 2 * lines[1]["gpu_launches"]
    tmp_path = tmp_path / "steps2"
    assert sorted(os.listdir(str(tmp_path))) == ["out.npy"]
    got = np.load(str(tmp_path / "out.npy"))
    import sr_wavenet_b200 as srwn
    from sr_wavenet_b200 import synth
    dil = synth.DEFAULT_DILATIONS
    s = srwn.ParallelWaveNet(T, 0, dil, None, num_flows=4, skip_channels=128, latent_channels=32, pool_stride=128)
    s.set_weights(synth.make_student_weights(dil, 4))
    ref = s.generate(None, synth.logistic_noise(B, T, seed=777), synth.synthetic_encoding(B, T // 128, seed=4321),
                     precision=d["config"]["precision_path"])
    assert got.dtype == np.float32 and got.shape == ref.shape == (B, T, 1)
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-6)
