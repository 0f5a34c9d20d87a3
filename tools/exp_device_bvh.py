"""Device BVH build against the host build on the dragon stand-in and the bunny.

Times (host clock, best of 3 after a warm-up call):
  host_build_ms          ct_host_build_bvh alone;
  device_build_call_ms   api.build_bvh: ct_gpu_build_bvh plus the wrapper's numpy arrays (host memory in, host memory out);
  device_build_laps_ms   CT_GPU_TIMING=1's laps inside one ct_gpu_build_bvh call (allocation, copies, the device build itself);
  upload_host_tree_ms    ct_gpu_upload_scene with the host-built tree, and its laps;
  upload_build_flag_ms   ct_gpu_upload_scene with CT_FLAG_BUILD_BVH (tree built in place, nothing back to the host), and its laps.
Checks that both trees are identical and that the first frame of both uploads hashes the same.  Prints the GPU's name and power
limit with the numbers.  Usage: python tools/exp_device_bvh.py [out.json]"""
import dataclasses
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cobbletrace_b200 as ct  # noqa: E402
from cobbletrace_b200 import api, host, procedural  # noqa: E402

TREE = ("node_min", "node_max", "node_left", "node_first", "node_count", "tri_index")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    return q.stdout.strip().splitlines()[0]


def best_ms(fn, reps=3):
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


def laps(fn):
    """fn() with CT_GPU_TIMING=1; returns {lap: ms} parsed from what the library prints on stderr."""
    os.environ["CT_GPU_TIMING"] = "1"
    with tempfile.TemporaryFile() as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["CT_GPU_TIMING"]
        f.seek(0)
        text = f.read().decode()
    return {m.group(1).strip(): float(m.group(2)) for m in re.finditer(r"^ct_gpu_\w+: (.+?)\s+([0-9.]+) ms$", text, re.M)}


def upload_ms(fs, build):
    r = ct.GpuRenderer(0)
    try:
        size = 640
        r.upload(fs, size, size, max_depth=10, build_bvh=build)                 # warm-up
        best = best_ms(lambda: r.upload(fs, size, size, max_depth=10, build_bvh=build))
        lap = laps(lambda: r.upload(fs, size, size, max_depth=10, build_bvh=build))
        r.render_tile()
        return best, lap, ct.frame_fnv1a(r.readback())
    finally:
        r.shutdown()


def measure(name, bare):
    """`bare`: a FlatScene without a tree.  The host build runs ct_host_build_bvh over the same triangles."""
    def host_build():                                                   # a scene keeps its tree: a fresh one per build, timed apart
        hs = host.HostScene.from_flat(bare)
        t0 = time.perf_counter()
        hs.build_bvh()
        return (time.perf_counter() - t0) * 1e3, hs
    host_build()                                                        # warm-up
    host_ms = min(host_build()[0] for _ in range(3))
    fs_host = dataclasses.replace(bare, **{k: getattr(host_build()[1].to_flat(with_bvh=True), k) for k in TREE})
    api.build_bvh(bare)                                                 # first call: module load
    dev_ms = best_ms(lambda: api.build_bvh(bare))
    dev_laps = laps(lambda: api.build_bvh(bare))
    fs_dev = api.build_bvh(bare)
    up_host, up_host_laps, frame_host = upload_ms(fs_host, False)
    up_flag, up_flag_laps, frame_flag = upload_ms(bare, True)
    row = dict(scene=name, n_tri=bare.n_tri, n_nodes=fs_host.n_nodes, host_cpus=os.cpu_count(), host_build_ms=round(host_ms, 2),
               device_build_call_ms=round(dev_ms, 2), device_build_laps_ms=dev_laps,
               upload_host_tree_ms=round(up_host, 2), upload_host_tree_laps_ms=up_host_laps,
               upload_build_flag_ms=round(up_flag, 2), upload_build_flag_laps_ms=up_flag_laps,
               identical_tree=fs_dev.bvh_digest() == fs_host.bvh_digest(), frame_host_tree=frame_host, frame_build_flag=frame_flag)
    print(json.dumps(row), flush=True)
    return row


def main():
    out = {"gpu": gpu_info()}
    print(out["gpu"], flush=True)
    with tempfile.TemporaryDirectory() as d:
        scene, _ = procedural.write_dragon_standin(d)
        dragon = host.HostScene.load(scene, base_dir=d).to_flat(with_bvh=False)
    bunny = ct.load_ctscene(os.path.join(ROOT, "tests", "golden", "scenes", "scene_import_bunny.ctscene.xz")).without_bvh()
    out["rows"] = [measure("dragon_standin", dragon), measure("scene_import_bunny", bunny)]
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)
    assert all(r["identical_tree"] and r["frame_host_tree"] == r["frame_build_flag"] for r in out["rows"])


if __name__ == "__main__":
    main()
