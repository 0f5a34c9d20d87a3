"""ct_gpu_update_triangles on bench.py's dragon4k workload and the bunny at 1080p, against a re-upload, and as one step of an animation.

Scenes: the dragon-class stand-in at 3840 x 2160 with depth 2 and reflection 0.5, built the way bench.py builds it (its load_host_scene),
and scene_import_bunny at 1920 x 1080 with depth 10 (bench.py's bunny1080).  Per scene, median of 7 after 2 warm-ups each:
  update           host clock around GpuRenderer.update_triangles (synchronous) with torch tensors already on the device, two deformed
                   meshes in turn (every call builds a different tree);
  re-upload        host clock around GpuRenderer.upload(..., build_bvh=True) of the same deformed meshes from host arrays -- the way to
                   move triangles before ct_gpu_update_triangles;
  animation step   a torch deformation on the current stream -> update_triangles -> render_tile of the whole frame -> sync, host clock;
  frame            ct_gpu_last_tile_ms of render_tile alone, for scale.
Then one update with CT_GPU_TIMING set: the library's own laps (host clock between its synchronisation points).  After the timings, the
frame of the last animation step is compared with a fresh upload of the same triangles.  Prints the GPU's name and power limit.
Usage: python tools/exp_update_triangles.py [out_prefix]  (writes out_prefix.json and out_prefix.txt)"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import cobbletrace_b200 as ct  # noqa: E402

REPS, WARM = 7, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    return q.stdout.strip().splitlines()[0]


def median_ms(call):
    for i in range(WARM):
        call(i)
    ms = []
    for i in range(REPS):
        t = time.perf_counter()
        call(WARM + i)
        ms.append((time.perf_counter() - t) * 1e3)
    return float(np.median(ms)), [round(v, 3) for v in ms]


def deform(t0, step):
    """A wave through the mesh, on the GPU (torch, current stream)."""
    import torch
    v = t0.view(-1, 3, 3)
    ext = (v.amax((0, 1)) - v.amin((0, 1))).clamp_min(1e-9)
    phase = (v - v.amin((0, 1))) / ext * 6.0 + 0.7 * step
    return (v + 0.01 * ext * torch.sin(phase[..., [1, 2, 0]])).reshape(-1, 9).contiguous()


def laps(r, t):
    """One update with CT_GPU_TIMING set: the library's lap lines (its stderr)."""
    with tempfile.TemporaryFile("w+") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        os.environ["CT_GPU_TIMING"] = "1"
        try:
            r.update_triangles(t)
        finally:
            del os.environ["CT_GPU_TIMING"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        return [line.rstrip() for line in f if line.startswith("ct_gpu_update_triangles")]


def measure(name, fs, W, H, depth):
    import dataclasses
    import torch
    r = ct.GpuRenderer(0)
    bare = fs.without_bvh()
    r.upload(bare, W, H, max_depth=depth, build_bvh=True)
    t0 = torch.from_numpy(np.ascontiguousarray(fs.tri, np.float64)).cuda()
    meshes = [deform(t0, k) for k in (1, 2)]
    host_meshes = [dataclasses.replace(bare, tri=m.cpu().numpy()) for m in meshes]
    torch.cuda.synchronize()
    row = dict(scene=name, frame=f"{W}x{H}", max_depth=depth, triangles=int(fs.n_tri))
    row["update_ms"], row["update_runs_ms"] = median_ms(lambda i: r.update_triangles(meshes[i % 2]))
    s = r.debug_scene_array("summary")
    row["depth"], row["n_pairs"], row["n_wide"] = int(s["depth"]), int(s["n_pairs"]), int(s["n_wide"])
    row["reupload_ms"], row["reupload_runs_ms"] = median_ms(lambda i: r.upload(host_meshes[i % 2], W, H, max_depth=depth, build_bvh=True))

    def step(i):
        r.update_triangles(deform(t0, i))
        r.render_tile()
        r.sync()
    row["animation_step_ms"], row["animation_step_runs_ms"] = median_ms(step)
    frame = r.readback().copy()
    tiles = []
    for _ in range(WARM + REPS):
        r.render_tile()
        tiles.append(r.last_tile_ms())
    row["frame_ms"] = round(float(np.median(tiles[WARM:])), 3)
    last = deform(t0, WARM + REPS - 1).cpu().numpy()
    r.upload(dataclasses.replace(bare, tri=last), W, H, max_depth=depth, build_bvh=True)
    r.render_tile()
    row["animation_frame_equals_fresh_upload"] = bool(np.array_equal(r.readback(), frame))
    row["laps"] = laps(r, meshes[0])
    r.shutdown()
    for k in ("update_ms", "reupload_ms", "animation_step_ms"):
        row[k] = round(row[k], 3)
    print(json.dumps(row), flush=True)
    return row


def main():
    out = {"gpu": gpu_info(), "timing": f"host clock around each synchronous call (animation step: deform, update, render, sync); median of "
           f"{REPS} after {WARM} warm-ups; frame: ct_gpu_last_tile_ms, the same median"}
    print(out["gpu"], flush=True)
    hs, _ = bench.load_host_scene("dragon", bench.REFLECTION)
    _, _, W, H, depth, _ = bench.WORKLOADS["dragon4k"]
    out["rows"] = [measure("dragon_standin", hs.to_flat(with_bvh=False), W, H, depth)]
    from conftest import load_golden_scene
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
    _, _, W, H, depth, _ = bench.WORKLOADS["bunny1080"]
    out["rows"].append(measure("scene_import_bunny", load_golden_scene("scene_import_bunny", golden), W, H, depth))
    if len(sys.argv) > 1:
        with open(sys.argv[1] + ".json", "w") as f:
            json.dump(out, f, indent=1)
        with open(sys.argv[1] + ".txt", "w") as f:
            f.write(f"ct_gpu_update_triangles -- {out['gpu']}; {out['timing']}\n")
            f.write("scene | frame | max_depth | triangles | tree depth | update ms | re-upload ms | animation step ms | frame ms | "
                    "animation frame equals a fresh upload\n")
            for r in out["rows"]:
                f.write(f"{r['scene']} | {r['frame']} | {r['max_depth']} | {r['triangles']} | {r['depth']} | {r['update_ms']} | "
                        f"{r['reupload_ms']} | {r['animation_step_ms']} | {r['frame_ms']} | {r['animation_frame_equals_fresh_upload']}\n")
            for r in out["rows"]:
                f.write(f"\nCT_GPU_TIMING laps, {r['scene']}:\n" + "\n".join(r["laps"]) + "\n")


if __name__ == "__main__":
    main()
