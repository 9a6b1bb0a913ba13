"""bench.py prints ONE JSON line with the keys the round driver reads (metric / value / e2e / roofline / cpu_baseline / clocks /
gpu_launches ...), for the product arm and for `--impl reference`."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _ref_kind():
    sys.path.insert(0, ROOT)
    from oracle import make_ref
    return "reference" if make_ref.available() else "port"


def test_product_arm_line(tmp_path):
    d = _run("--steps", "4", "--warmup", "3", "--sustain", "1.0", "--dump-outputs", str(tmp_path))
    assert d["metric"] == "images/sec (backbone+decode)" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] == 3 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "bf16" and d["data"] == "synthetic" and "BASELINE configs[1]" in d["config"]["workload"]
    assert d["value"] > 1000 and abs(d["ms_per_step"] * d["value"] / 1e3 - 64) < 0.5          # 64 images per step
    e = d["e2e"]
    assert e["unit"] == "images/sec" and 0 < e["value"] <= d["value"] * 1.05
    assert e["h2d_bytes_per_step"] == 64 * 513 * 513 * 3 and e["d2h_bytes_per_step"] == 64 * 10 * 86 * 8
    assert d["gpu_launches"] >= 15 * 4
    c = d["clocks"]
    assert c["sm_mhz"] and c["sm_max_mhz"] and isinstance(c["reasons"], list) and c["samples_in_timed_region"] >= 1
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert 0 < r["frac"] <= 1.0
    b = d["cpu_baseline"]
    assert b["kind"] == _ref_kind() and b["cores"] >= 1 and b["value"] > 0 and b["sample"]
    assert abs(sum(k["share"] for k in d["kernels"]) - 1.0) < 0.01
    # the ceiling the host can feed, and the end-to-end figure as a fraction of it
    assert e["h2d_ceiling_gbs"] > 0 and 0 < e["frac_of_h2d_ceiling"] < 1.2
    # sustained leg: the same replays for ~1 s here (3 s by default), with its own clock samples
    su = d["sustained"]
    assert d["value_sustained"] == su["value"] and su["seconds"] >= 0.9 and 0.3 < su["vs_burst"] < 1.2
    assert su["clocks"]["sm_mhz"] and isinstance(su["clocks"]["reasons"], list)
    assert d["run"]["batch_per_gpu"] == 64 and d["config"]["model"] == "mobilenet_v1_101"
    # --dump-outputs: the records of the last timed step (step 3 of 4 reads input set 3), float64, equal to an eager run of
    # the same seeded model on the same seeded images
    sys.path.insert(0, ROOT)
    import bench
    import posenet
    import torch
    dumped = [np.load(tmp_path / (name + ".npy")) for name in bench.DUMP_NAMES]
    assert sorted(os.listdir(tmp_path)) == sorted(name + ".npy" for name in bench.DUMP_NAMES)
    assert all(a.dtype == np.float64 for a in dumped) and dumped[2].shape == (64, 10, 17, 2)
    rng = np.random.default_rng(1234)
    x = [rng.integers(0, 256, (64, 513, 513, 3), dtype=np.uint8) for _ in range(4)][3]
    torch.manual_seed(0)
    model = posenet.MobileNetV1(101, output_stride=16).cuda().set_compute_dtype("bf16").set_fused(True)
    ref = posenet.decode_multiple_poses_batch(*model.forward_u8(torch.from_numpy(x).cuda()), output_stride=16, **bench.DECODE_KW)
    for a, b in zip(dumped, ref):
        assert np.array_equal(a, b.cpu().numpy().astype(np.float64))
    assert np.array_equal(dumped[4], (dumped[0] != 0).sum(1))


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert d["impl"] == "reference" and d["metric"] == "images/sec (backbone+decode)" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == _ref_kind() and d["cpu_baseline"]["value"] == d["value"]
    # both arms describe the same workload: the config objects are identical (how each arm batches it is under "run")
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config("c2") and d["run"]["batch"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
