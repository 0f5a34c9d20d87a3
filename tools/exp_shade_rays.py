"""ct_gpu_shade_rays on bench.py's dragon4k workload and the bunny at 1080p, against the frame that shades the same rays.

Scenes: the dragon-class stand-in at 3840 x 2160 with depth 2 and reflection 0.5, built the way bench.py builds it (its
load_host_scene), and scene_import_bunny at 1920 x 1080 with depth 10 (bench.py's bunny1080).  Workloads per scene, the rays in device
memory, CUDA events on torch's current stream around one call, median of 7 after 2 warm-up calls, best of 3 rounds; the scene's arrays
stay in L2 between calls, the rays stream through:
  camera scanline   the frame's own camera rays (the centred H x H square), row by row;
  camera blocks     the same rays in the frame's slot order (8 x 4 pixel blocks);
  camera random     the same rays in a random order;
  random 1k / 64k   the first 1 k / 64 k random-order rays: the fixed cost of a call.
Beside them: ct_gpu_last_tile_ms of the frame (render_tile, the same median), and whether the scanline colours equal its pixels.
Prints the GPU's name and power limit.  Usage: python tools/exp_shade_rays.py [out.json]"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import cobbletrace_b200 as ct  # noqa: E402
from test_shade_rays import canvas_rays, frame_pixels  # noqa: E402

REPS, WARM = 7, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    return q.stdout.strip().splitlines()[0]


def median_ms(call):
    import torch
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(WARM):
        call()
    ms = []
    for _ in range(REPS):
        ev[0].record()
        call()
        ev[1].record()
        ev[1].synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return float(np.median(ms))


def tile_ms(r):
    ms = []
    for _ in range(WARM + REPS):
        r.render_tile()
        ms.append(r.last_tile_ms())
    return float(np.median(ms[WARM:]))


def measure(name, fs, W, H, depth):
    import torch
    r = ct.GpuRenderer(0)
    r.upload(fs, W, H, max_depth=depth)
    frame_ms = min(tile_ms(r) for _ in range(3))
    frame = r.readback()
    x, y, row, col, blocks = frame_pixels(W, H)
    o, d = canvas_rays(fs, H, x, y)
    ot, dt = (torch.from_numpy(a).cuda() for a in (o, d))
    same = bool(np.array_equal(r.shade_rays(ot, dt).cpu().numpy().view(np.uint32), frame[row, col]))
    b = torch.from_numpy(blocks).cuda()
    perm = torch.randperm(len(o), generator=torch.Generator().manual_seed(1)).cuda()
    rp = ot[perm].contiguous(), dt[perm].contiguous()
    work = {"camera scanline": (ot, dt), "camera blocks": (ot[b].contiguous(), dt[b].contiguous()), "camera random": rp,
            "random 1k": (rp[0][:1024].contiguous(), rp[1][:1024].contiguous()),
            "random 64k": (rp[0][:65536].contiguous(), rp[1][:65536].contiguous())}
    rows = []
    for wl, (a, e) in work.items():
        runs = [median_ms(lambda: r.shade_rays(a, e)) for _ in range(3)]
        row_ = dict(scene=name, frame=f"{W}x{H}", max_depth=depth, workload=wl, rays=int(a.shape[0]), ms=round(min(runs), 3),
                    runs_ms=[round(v, 3) for v in runs])
        print(json.dumps(row_), flush=True)
        rows.append(row_)
    r.shutdown()
    summary = dict(scene=name, frame=f"{W}x{H}", max_depth=depth, rays=len(o), last_tile_ms=round(frame_ms, 3), scanline_equals_frame=same)
    print(json.dumps(summary), flush=True)
    return rows, summary


def main():
    out = {"gpu": gpu_info(), "timing": f"CUDA events around one call on torch's current stream; median of {REPS} after {WARM} warm-up "
           f"calls, best of 3 rounds; L2 warm (scene arrays resident, rays streamed); frames: ct_gpu_last_tile_ms, the same median"}
    print(out["gpu"], flush=True)
    hs, _ = bench.load_host_scene("dragon", bench.REFLECTION)
    _, _, W, H, depth, _ = bench.WORKLOADS["dragon4k"]
    out["rows"], out["frames"] = [], []
    rows, summary = measure("dragon_standin", hs.to_flat(with_bvh=True), W, H, depth)
    out["rows"] += rows; out["frames"].append(summary)
    from conftest import load_golden_scene
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
    _, _, W, H, depth, _ = bench.WORKLOADS["bunny1080"]
    rows, summary = measure("scene_import_bunny", load_golden_scene("scene_import_bunny", golden), W, H, depth)
    out["rows"] += rows; out["frames"].append(summary)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
