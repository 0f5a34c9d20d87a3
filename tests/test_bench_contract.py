"""bench.py's contract, as far as it can be checked without a GPU: the reference arm prints one JSON line with the agreed
keys (the compiled reference on host cores, on the small configs[0] workload here), and the GPU arm refuses to run
without a CUDA device instead of measuring anything on the CPU."""
import json
import os
import subprocess
import sys

import pytest

from oracle import ct_oracle_py as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/ct_ref not built (needs the reference's sources once: CT_REFERENCE_SRC)")
def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cube640", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]
    # the reference arm names the workload exactly as the GPU arm does (same function, same keys), with the scene's sizes
    # taken from the reference's own run, and loads nothing of the product while it measures
    import bench
    assert d["config"] == bench.workload_config("cube640", 1, 37, 15, 3)
    assert d["rays_per_step"] == {"rays_primary": 409600, "rays_shadow": 1516008, "rays_reflection": 348404}       # SURVEY section 6 (reference counters)
    src = open(os.path.join(ROOT, "bench.py")).read()
    arm = src[src.index("def reference_arm"):src.index("# ---- our arm")]
    assert "from cobbletrace_b200 import host" not in arm.split("else:")[0]


def test_bench_frame_pins_are_what_the_oracle_renders(golden, scene_loader):
    """tests/golden/bench_frames.json (hashes of the bench workloads' frames from the compiled reference) against the oracle
    on the same inputs, for the workloads the oracle finishes in seconds."""
    import bench
    from cobbletrace_b200.sceneio import frame_fnv1a
    pins = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_frames.json")))
    assert set(pins) >= {"dragon4k", "dragon8k", "cube640", "import640", "bunny1080", "pcbig1080"}
    for key, scene in (("cube640", "scene_file_cube"), ("import640", "scene_import")):
        desc, kind, W, H, depth, refl = bench.WORKLOADS[key][:6]
        frame, _, _ = O.OracleScene(scene_loader(scene)).render(W, H, max_depth=depth, want_hits=False)
        assert frame_fnv1a(frame) == pins[key]["fnv1a"] == golden["scenes"][scene]["frame640_fnv1a"], key
        assert bench.expected_frame(key)[0] == pins[key]["fnv1a"]


def test_gpu_arm_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cube640", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
    assert not [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]          # and prints no result line
