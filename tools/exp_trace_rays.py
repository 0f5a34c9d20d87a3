"""ct_gpu_trace_rays on the dragon stand-in and the bunny, with the rays in the caller's order (default build) and binned (a second
libct_gpu.so built here with -DCT_RAY_BINS=1), alternating.

Workloads per scene (rays in device memory, CUDA events on torch's current stream around one call, median of 7 after 2 warm-up
calls; the scene's arrays stay in L2 between calls -- the dragon's 76 MB hot set fits the 126 MB -- the rays stream through):
  primary pixel     CT_RAY_PRIMARY, the 4K camera's primary rays (the centred 2160 x 2160 square: 4.67 M) in scanline order;
  primary random    the same rays in a random order;
  shadow ao         CT_RAY_SHADOW, 8 seeded hemisphere directions per primary hit point (at most 2^21 hit points);
  reflection        CT_RAY_REFLECTION from the hit points, mirrored about the triangle's normal;
  primary 1k / 64k  the first 1 k / 64 k random-order primary rays: the fixed cost of a call.
Beside them: k_primary's own stage time for the same frame (CT_FLAG_STAGE_TIMING, max_depth 0, pixel blocks of 8 x 4).
Checks that both builds give the same bits.  Prints the GPU's name and power limit.  Usage: python tools/exp_trace_rays.py [out.json]"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cobbletrace_b200 as ct  # noqa: E402
from cobbletrace_b200 import api, build, host, procedural  # noqa: E402

W, H = 3840, 2160
REPS, WARM = 7, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    return q.stdout.strip().splitlines()[0]


def build_binned(d):
    lib = os.path.join(d, "libct_gpu_bins1.so")
    src = os.path.join(build.CSRC, "ct_gpu.cu")
    subprocess.check_call([build.find_nvcc()] + build.NVCC_FLAGS + ["-DCT_RAY_BINS=1", "-o", lib, src], cwd=ROOT)
    return lib


def camera_rays(fs):
    """The primary rays of the W x H frame's centred square, scanline order (primary_ray_at's arithmetic)."""
    half = H // 2
    s = np.float64(np.float32(1.0) / np.float32(H))
    ys, xs = np.meshgrid(np.arange(half, half - H, -1, dtype=np.float64), np.arange(-half, half, dtype=np.float64), indexing="ij")
    v = np.stack([xs.ravel() * s, ys.ravel() * s, np.ones(xs.size)], 1)
    rot = np.asarray(fs.cam_rot, np.float64).reshape(3, 3)
    d = v @ rot
    o = np.broadcast_to(np.asarray(fs.cam_pos, np.float64), d.shape).copy()
    return o, d


def time_call(r, o, d, kind):
    import torch
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(WARM):
        r.trace_rays(o, d, kind)
    ms = []
    for _ in range(REPS):
        ev[0].record()
        out = r.trace_rays(o, d, kind)
        ev[1].record()
        ev[1].synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return float(np.median(ms)), out


def k_primary_ms(fs):
    r = ct.GpuRenderer(0)
    try:
        r.upload(fs, W, H, max_depth=0, flags=api.CT_FLAG_STAGE_TIMING)
        best = []
        for _ in range(WARM + REPS):
            r.render_tile()
            best.append(sum(ms for name, _, ms in r.last_tile_stages() if name == "primary"))
        return float(np.median(best[WARM:]))
    finally:
        r.shutdown()


def workloads(fs, r):
    import torch
    o, d = camera_rays(fs)
    ot, dt = (torch.from_numpy(x).cuda() for x in (o, d))
    perm = torch.randperm(len(o), generator=torch.Generator().manual_seed(1)).cuda()
    f, i, t = r.trace_rays(ot, dt, "primary")
    hit = torch.nonzero(f != 0).squeeze(1)[: 1 << 21]
    tri = torch.from_numpy(np.ascontiguousarray(fs.tri, np.float64).reshape(-1, 3, 3)).cuda()[i[hit].long()]
    n = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    n = n / n.norm(dim=1, keepdim=True)
    dh = dt[hit]
    n = torch.where(((n * dh).sum(1, keepdim=True) > 0), -n, n)                    # towards the camera
    p = ot[hit] + t[hit].double().unsqueeze(1) * dh
    g = torch.Generator(device="cuda").manual_seed(2)
    a = torch.randn((len(hit), 8, 3), generator=g, device="cuda", dtype=torch.float64)
    a = torch.where(((a * n.unsqueeze(1)).sum(2, keepdim=True) < 0), -a, a)        # the hemisphere about n
    refl = dh - 2.0 * (dh * n).sum(1, keepdim=True) * n
    rp = ot[perm].contiguous(), dt[perm].contiguous()
    return {
        "primary pixel": ("primary", ot, dt),
        "primary random": ("primary",) + rp,
        "shadow ao": ("shadow", p.repeat_interleave(8, 0).contiguous(), a.reshape(-1, 3).contiguous()),
        "reflection": ("reflection", p.contiguous(), refl.contiguous()),
        "primary 1k": ("primary", rp[0][:1024].contiguous(), rp[1][:1024].contiguous()),
        "primary 64k": ("primary", rp[0][:65536].contiguous(), rp[1][:65536].contiguous()),
    }


def measure(name, fs, lib1):
    import torch
    binned = ct.GpuRenderer(0)
    caller = ct.GpuRenderer(0)
    binned.L = api.load_library(lib1)
    binned.upload(fs, 64, 64, max_depth=2)
    caller.upload(fs, 64, 64, max_depth=2)
    rows = []
    for wl, (kind, o, d) in workloads(fs, caller).items():
        t = {"binned": [], "caller_order": []}
        outs = {}
        for _ in range(3):                                                          # alternate the two builds
            for tag, r in (("binned", binned), ("caller_order", caller)):
                ms, out = time_call(r, o, d, kind)
                t[tag].append(ms)
                outs[tag] = out
        same = all((a is None and b is None) or torch.equal(a, b) for a, b in zip(outs["binned"], outs["caller_order"]))
        row = dict(scene=name, workload=wl, kind=kind, rays=int(o.shape[0]), binned_ms=round(min(t["binned"]), 3),
                   caller_order_ms=round(min(t["caller_order"]), 3), binned_runs_ms=[round(x, 3) for x in t["binned"]],
                   caller_order_runs_ms=[round(x, 3) for x in t["caller_order"]], identical_results=bool(same))
        row["binned_mrays_s"] = round(row["rays"] / row["binned_ms"] / 1e3, 1)
        row["caller_order_mrays_s"] = round(row["rays"] / row["caller_order_ms"] / 1e3, 1)
        print(json.dumps(row), flush=True)
        rows.append(row)
    caller.shutdown()
    binned.L.ct_gpu_shutdown(0)
    return rows, k_primary_ms(fs)


def main():
    out = {"gpu": gpu_info(), "frame": f"{W}x{H}", "timing": f"CUDA events around one call on torch's current stream; median of {REPS} "
           f"after {WARM} warm-up calls, best of 3 alternating rounds; L2 warm (scene arrays resident, rays streamed)"}
    print(out["gpu"], flush=True)
    with tempfile.TemporaryDirectory() as d:
        lib1 = build_binned(d)
        path, _ = procedural.write_dragon_standin(d)
        dragon = api.build_bvh(host.HostScene.load(path, base_dir=d).to_flat(with_bvh=False))
        bunny = api.build_bvh(ct.load_ctscene(os.path.join(ROOT, "tests", "golden", "scenes", "scene_import_bunny.ctscene.xz")).without_bvh())
        out["rows"], out["k_primary_stage_ms"] = [], {}
        for name, fs in (("dragon_standin", dragon), ("scene_import_bunny", bunny)):
            rows, kp = measure(name, fs, lib1)
            out["rows"] += rows
            out["k_primary_stage_ms"][name] = round(kp, 3)
            print(json.dumps({"scene": name, "k_primary_stage_ms": round(kp, 3)}), flush=True)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)
    assert all(r["identical_results"] for r in out["rows"])


if __name__ == "__main__":
    main()
