"""ct_gpu_update_scene on bench.py's dragon4k workload (the dragon-class stand-in at 3840 x 2160, depth 2, reflection 0.5, built the way
bench.py builds it), against what a caller has without it: copying the same data to the host and re-uploading with CT_FLAG_BUILD_BVH.

Edits, each alternating between two versions already in device memory (torch tensors), so that every call changes the scene:
  materials   new colours, speculars and reflections for every triangle (update_scene(materials=...): no tree rebuild);
  lights      the 3 lights moved and re-coloured in intensity (update_scene(lights=...));
  count       the mesh and a copy without its last 10 % of triangles, with their materials (update_scene(triangles=, materials=)).
Per edit: host clock around the synchronous update_scene call, and around the re-upload (tensors copied to the host, then
GpuRenderer.upload(..., build_bvh=True)); median of 7 after 2 warm-ups.  After the timings, the frame rendered after the last update is
compared with a fresh upload of the same scene, and the frame time (ct_gpu_last_tile_ms, median of 7) is taken.  Records the GPU's name
and power limit.
Usage: python tools/exp_update_scene.py [out_prefix]  (default profiles/r07_update_scene; writes out_prefix.json and out_prefix.txt)"""
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
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
    return round(float(np.median(ms)), 3), [round(v, 3) for v in ms]


def main():
    import torch
    prefix = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_update_scene")
    out = {"gpu": gpu_info(), "timing": f"host clock around each synchronous call; median of {REPS} after {WARM} warm-ups"}
    print(out["gpu"], flush=True)
    hs, _ = bench.load_host_scene("dragon", bench.REFLECTION)
    _, _, W, H, depth, _ = bench.WORKLOADS["dragon4k"]
    fs = hs.to_flat(with_bvh=False)
    rng = np.random.default_rng(7)
    dev = torch.device("cuda", 0)
    n = fs.n_tri
    k = n - n // 10
    gpu = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)

    def mats(color, spec, refl):
        return (gpu(color, np.uint32).to(torch.int64), gpu(spec, np.int32), gpu(refl, np.float32))

    def lights(f):
        return (gpu(f.light_type, np.int32), gpu(f.light_intensity, np.float32), gpu(f.light_pos, np.float64), gpu(f.light_dir, np.float64))

    mat_sets = [mats(fs.mat_color, fs.mat_specular, fs.mat_reflection),
                mats(rng.integers(0, 1 << 24, n).astype(np.uint32), rng.choice(np.array([-1, 10, 500], np.int32), n),
                     np.full(n, 0.25, np.float32))]
    moved = dataclasses.replace(fs, light_pos=fs.light_pos + rng.normal(size=fs.light_pos.shape),
                                light_intensity=(fs.light_intensity * 0.9).astype(np.float32))
    light_sets = [lights(fs), lights(moved)]
    tri_sets = [(gpu(fs.tri, np.float64), mat_sets[0]), (gpu(fs.tri[:k], np.float64), tuple(a[:k] for a in mat_sets[0]))]
    torch.cuda.synchronize()

    def host_scene(tri=None, m=None, lt=None):
        """The scene a re-upload needs, with the edited parts copied back from the device."""
        f = fs
        if tri is not None:
            f = dataclasses.replace(f, tri=tri.cpu().numpy())
        if m is not None:
            f = dataclasses.replace(f, mat_color=(m[0].cpu().numpy() & 0xFFFFFFFF).astype(np.uint32), mat_specular=m[1].cpu().numpy(),
                                    mat_reflection=m[2].cpu().numpy())
        if lt is not None:
            f = dataclasses.replace(f, light_type=lt[0].cpu().numpy(), light_intensity=lt[1].cpu().numpy(), light_pos=lt[2].cpu().numpy(),
                                    light_dir=lt[3].cpu().numpy())
        return f

    edits = {
        "materials": (lambda i: dict(materials=mat_sets[i % 2]), lambda i: host_scene(m=mat_sets[i % 2])),
        "lights": (lambda i: dict(lights=light_sets[i % 2]), lambda i: host_scene(lt=light_sets[i % 2])),
        "count": (lambda i: dict(triangles=tri_sets[i % 2][0], materials=tri_sets[i % 2][1]),
                  lambda i: host_scene(tri=tri_sets[i % 2][0], m=tri_sets[i % 2][1])),
    }
    r = ct.GpuRenderer(0)
    out["scene"] = dict(name="dragon_standin", frame=f"{W}x{H}", max_depth=depth, triangles=int(n), triangles_after_count_edit=int(k),
                        lights=int(fs.n_lights))
    out["rows"] = []
    for name, (args, scene) in edits.items():
        r.upload(fs, W, H, max_depth=depth, build_bvh=True)
        row = dict(edit=name)
        row["update_ms"], row["update_runs_ms"] = median_ms(lambda i: r.update_scene(**args(i)))
        last = scene(WARM + REPS - 1)
        r.render_tile()
        frame = r.readback().copy()
        tiles = []
        for _ in range(WARM + REPS):
            r.render_tile()
            tiles.append(r.last_tile_ms())
        row["frame_ms_after"] = round(float(np.median(tiles[WARM:])), 3)
        row["reupload_ms"], row["reupload_runs_ms"] = median_ms(lambda i: r.upload(scene(i), W, H, max_depth=depth, build_bvh=True))
        r.upload(last, W, H, max_depth=depth, build_bvh=True)
        r.render_tile()
        row["frame_equals_fresh_upload"] = bool(np.array_equal(r.readback(), frame))
        print(json.dumps(row), flush=True)
        out["rows"].append(row)
    r.shutdown()
    with open(prefix + ".json", "w") as f:
        json.dump(out, f, indent=1)
    with open(prefix + ".txt", "w") as f:
        s = out["scene"]
        f.write(f"ct_gpu_update_scene -- {out['gpu']}; {out['timing']}\n")
        f.write(f"{s['name']} {s['frame']} depth {s['max_depth']}, {s['triangles']} triangles ({s['triangles_after_count_edit']} after the "
                f"count edit), {s['lights']} lights\n")
        f.write("edit | update_scene ms | host copy + re-upload ms | frame ms after the update | frame equals a fresh upload\n")
        for row in out["rows"]:
            f.write(f"{row['edit']} | {row['update_ms']} | {row['reupload_ms']} | {row['frame_ms_after']} | {row['frame_equals_fresh_upload']}\n")


if __name__ == "__main__":
    main()
