"""The bench.py JSON-line contract, checked on the committed lines of the last GPU run (profiles/): every key the
driver reads is present and internally consistent.  (bench.py itself needs a B200; this guards the schema.)"""
import json
import os

import pytest

PROF = os.path.join(os.path.dirname(os.path.dirname(__file__)), "profiles")


def _load(name):
    path = os.path.join(PROF, name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not committed")
    return json.load(open(path))


def test_device_arm_line():
    d = _load("r02_bench_default.json")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["metric"] == "4-step 16x320x512 frames/sec" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["dtype"] == "bf16" and d["data"] == "synthetic" and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    # value = 16 frames per video x videos per step per GPU / device time
    bs = d["config"].get("videos_per_step") or int(d["config"]["workload"].split("bs=")[1].split()[0])
    assert abs(d["value"] - 16 * bs * d["n_gpus"] / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["unit"] == "frames/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == bs * 16 * 3 * 320 * 512 * 2
    assert e["value"] < d["value"]  # copies inside the timed region: never just a repeat of the device-timed number
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert not bad & set(d["clocks"]["reasons"])


def test_reference_arm_line():
    d = _load("r02_bench_reference_arm.json")
    assert d["impl"] == "reference" and d["metric"] == "4-step 16x320x512 frames/sec" and d["unit"] == "frames/s"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["config"]["workload"] == _load("r02_bench_default.json")["config"]["workload"]   # the same workload as our arm


def test_two_gpu_line_is_weak_scaling_aggregate():
    one, two = _load("r02_bench_default.json"), _load("r02_bench_2gpu.json")
    assert two["n_gpus"] == 2 and two["scaling"] == "weak"
    assert 1.8 < two["value"] / one["value"] < 2.2


def test_dump_outputs_sample_is_fixed_and_within_budget(tmp_path):
    """bench.py --dump-outputs: float32 / float64 files, small arrays whole, a large one as the same seeded sample every time,
    everything within the byte budget."""
    import numpy as np
    import torch

    import bench
    arrays = dict(video=torch.arange(3000.0).reshape(3, 1000), loss=torch.tensor([0.5], dtype=torch.bfloat16),
                  index=torch.tensor([7, 9]), w=torch.tensor([2.5], dtype=torch.float64))
    a, b = bench.snapshot_outputs(arrays, budget=4000), bench.snapshot_outputs(arrays, budget=4000)
    assert list(a) == list(arrays)
    assert {k: v.dtype for k, v in a.items()} == dict(video=np.float32, loss=np.float32, index=np.float64, w=np.float64)
    assert a["index"].tolist() == [7, 9] and a["w"].tolist() == [2.5] and a["loss"].shape == (1,)
    assert sum(v.nbytes for v in a.values()) <= 4000 and 0 < a["video"].size < 3000
    assert np.array_equal(a["video"], b["video"])
    assert np.all(np.diff(a["video"]) > 0) and np.all(a["video"] == np.round(a["video"]))   # ascending positions of the flattened array
    bench.write_outputs(str(tmp_path / "out"), a)
    assert sorted(os.listdir(tmp_path / "out")) == ["index.npy", "loss.npy", "video.npy", "w.npy"]
    assert np.array_equal(np.load(tmp_path / "out" / "video.npy"), a["video"])
