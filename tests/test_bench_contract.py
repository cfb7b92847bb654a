"""bench.py's reference arm runs without a GPU: check that it prints exactly ONE JSON line with the contract's keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "frames/s"
    assert d["metric"] == "rgbd_480x640_frames_per_sec_depth_guidance_hot_path"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "e2e",
                "cpu_baseline", "gpu_launches"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # `value` = the hot path alone, `e2e` = the whole model + post-processing on the CPU (like with like against the own
    # arm's two numbers); nothing crosses a host<->device link on this arm
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert 0 < e["value"] < d["value"]                              # the whole model is slower than its hot path
    assert d["value"] > 0 and "workload" in d["config"] and "model" not in d["config"]


import numpy as np  # noqa: E402
import pytest  # noqa: E402
import torch  # noqa: E402


def test_dump_outputs_keeps_to_64_mb_and_stores_the_same_elements_every_run(tmp_path):
    """--dump-outputs: float32 files, at most 64 MB in all; maps that fit whole, larger ones as a fixed sample.  Each map holds
    its own flat indices, so a sample shows which elements it kept."""
    import bench
    B = 8
    fused = [torch.arange(B * c * (bench.H // s) * (bench.W // s), dtype=torch.float32).view(B, c, bench.H // s, bench.W // s)
             for c, s in zip(bench.CHANS, bench.STRIDES)]
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), fused)
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == [f"fused{i}.npy" for i in range(4)]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 * 10**6
    whole = []
    for i, t in enumerate(fused):
        a, b = np.load(tmp_path / "a" / f"fused{i}.npy"), np.load(tmp_path / "b" / f"fused{i}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        whole.append(a.shape == tuple(t.shape))
        if whole[-1]:
            assert np.array_equal(a, t.numpy())
        else:
            assert a.ndim == 1 and 0 < a.size < t.numel() and (np.diff(a) > 0).all() and 0 <= a[0] and a[-1] < t.numel()
    assert whole == [False, False, True, True]


@pytest.mark.gpu
def test_own_arm_prints_one_contract_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--batch", "4",
                        "--cpu-steps", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["metric"] == "rgbd_480x640_frames_per_sec_depth_guidance_hot_path" and d["unit"] == "frames/s"
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "bf16" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["gpu_launches"] > 0 and "workload" in d["config"] and "model" not in d["config"]
    e = d["e2e"]
    assert e["value"] > 0 and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert e["value"] < d["value"]                                   # host copies are inside the e2e timed region
    rf = d["roofline"]
    assert rf["bound"] in ("hbm", "tensor") and rf["unit"] in ("GB/s", "TFLOP/s") and rf["peak"] > 0
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9 and "traffic" in rf
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    ck = d["clocks"]
    assert ck["sm_mhz"] > 0 and ck["sm_max_mhz"] >= ck["sm_mhz"] and isinstance(ck["reasons"], list)
    assert "RgbdInstanceSegmenter" in e["how"] and 0 < e["hot_path_share_of_step"] < 1
    hp = d["e2e_hot_path_host_features"]
    assert hp["check"]["bit_identical_to_device_resident_step"] is True and hp["value"] > 0
    tr = d["train"]
    assert tr["value"] > 0 and tr["batch_per_gpu"] == 8 and tr["ms_per_step"] > 0
    assert cb["detail"]["hot_path_1_thread_frames_per_s"] > 0 and cb["detail"]["whole_model_plus_postprocess_frames_per_s"] > 0
    # --dump-outputs: the last timed step's four fused maps (batch 4: the largest as a sample, the others whole)
    dumped = [np.load(tmp_path / f"fused{i}.npy") for i in range(4)]
    assert [a.shape for a in dumped[1:]] == [(4, c, 480 // s, 640 // s) for c, s in ((192, 8), (384, 16), (768, 32))]
    assert dumped[0].ndim == 1 and all(a.dtype == np.float32 and np.isfinite(a).all() for a in dumped)
