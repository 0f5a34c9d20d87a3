#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

metric   Mrays/s (primary + shadow + reflection rays, also reported by kind) and ms/frame
workload configs[2]: dragon-class scene (procedural 868 352-triangle stand-in for the missing dragon.ply,
         SURVEY 8d) at 3840x2160, shadow rays + 2 reflection bounces (maxDepth 2, reflection forced to 0.5)
step     one frame: every row tile of the frame through the hot path
value    device-resident throughput (scene in HBM, CUDA events around the frame's kernels [+ gather at N>1])
e2e      the same frame through the reference-facing plugin call with HOST buffers: camera in
         (ct_gpu_set_camera), bitmap out (ct_gpu_readback into pinned host memory), wall clock
N > 1    one process per GPU (torchrun), scene replicated; all GPUs render the same frame in 32-pixel chunks (7/8 dealt
         round-robin, 1/8 stolen from one cursor on GPU 0 with atomics over NVLink) and store finished pixels straight
         into GPU 0's framebuffer (peer stores); strong scaling of the same frame
--impl reference   the reference's own boss/worker CPU renderer (oracle/_ref/ct_ref, compiled from the unmodified
         sources) on this box's host cores, same scene files, same metric.
--dump-outputs DIR the frame the last timed step rendered, as DIR/frame.npy (see dump_frame), so that two builds can be
         compared pixel for pixel on the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s (primary+shadow+reflection) dragon-class 4K, shadows + 2 reflection bounces"


def metric_name(workload_key: str) -> str:
    return METRIC if workload_key.startswith("dragon") else f"Mrays/s (primary+shadow+reflection), workload {workload_key}"


def data_note(kind: str) -> str:
    if kind == "dragon":
        return "synthetic (procedural 868352-triangle octa-sphere stand-in for the missing dragon.ply, generated in-run)"
    return "bundled reference scene (tests/golden flattened copy of the reference's own scene file and meshes)"
REFLECTION = 0.5

WORKLOADS = {
    # name: (description, generator, width, height, max_depth, forced reflection)
    "dragon4k": ("configs[2]: dragon-class procedural stand-in (868352 tris, scene_import_dragon.json lights/camera/material), "
                 "3840x2160 (traced square 2160^2), shadows + 2 reflection bounces", "dragon", 3840, 2160, 2, REFLECTION),
    "dragon8k": ("configs[4]: same scene at 7680x4320 (traced square 4320^2)", "dragon", 7680, 4320, 2, REFLECTION),
    "dragon1080": ("reduced sample of configs[2]: same scene at 1920x1080", "dragon", 1920, 1080, 2, REFLECTION),
    "dragon1080ss": ("stress: the configs[2] scene at 1920x1080 with settings.supersampling (16 jittered samples per pixel, counter-based jitter)",
                     "dragon", 1920, 1080, 2, REFLECTION, 32),
    # the other BASELINE configs (parity-test cases; here for measurement on request, never the default)
    "cube640": ("configs[0]: scene_file_cube.json (37 triangles, 3 lights, one mirror) 640x640, depth 10", "golden:scene_file_cube", 640, 640, 10, None),
    "import640": ("configs[0]: scene_import.json (roundedCube.obj x4, 1712 triangles) 640x640, depth 10", "golden:scene_import", 640, 640, 10, None),
    "bunny1080": ("configs[1]: scene_import_bunny.json (69451 triangles) 1920x1080 (traced square 1080^2), shadow rays", "golden:scene_import_bunny", 1920, 1080, 10, None),
    "pcbig1080": ("configs[3]: utils/pc_big.json (6468 triangles, 66 lights from sphereOfLights) 1920x1080, any-hit bound", "golden:pc_big", 1920, 1080, 10, None),
}
GOLDEN_JSON = {"scene_file_cube": "scene_file_cube.json", "scene_import": "scene_import.json", "scene_import_bunny": "scene_import_bunny.json",
               "pc_big": "pc_big.json"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload_config(key: str, n_gpus: int, n_tri: int, n_nodes: int, n_lights: int) -> dict:
    """`config` of the JSON line: what was rendered.  The same function serves both arms, so that the two lines name the
    workload identically (how each arm ran it is in `method` / `cpu_baseline.sample`, not here)."""
    desc, kind, W, H, depth, refl = WORKLOADS[key][:6]
    return {"workload": desc, "scene": kind, "width": W, "height": H, "triangles": int(n_tri), "bvh_nodes": int(n_nodes), "lights": int(n_lights),
            "max_depth": depth, "forced_reflection": refl, "n_gpus": int(n_gpus),
            "l2": "b200 arm: flushed between timed steps (256 MiB device write, outside the timed events); reference arm: host CPU, not applicable"}


def expected_frame(key: str):
    """(fnv1a, source) of the workload's frame as the compiled, unmodified reference rendered it (tests/golden/bench_frames.json,
    made by tests/golden/make_golden_bench.py), or (None, None)."""
    try:
        e = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_frames.json")))[key]
        return e["fnv1a"], e["source"]
    except Exception:
        return None, None


def scene_cache_dir() -> str:
    d = os.environ.get("CT_SCENE_CACHE") or os.path.join("/tmp", f"ct_bench_scene_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def ensure_scene(kind: str):
    """(scene file the reference's parser can read, triangle count).  dragon: generated; golden:<name>: the reference's own
    scene file as copied next to the compiled reference (oracle/_ref/scenes), triangle count from tests/golden."""
    from cobbletrace_b200 import procedural
    if kind == "dragon":
        return procedural.write_dragon_standin(scene_cache_dir())
    from oracle import ct_oracle_py as O
    name = kind.split(":", 1)[1]
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["scenes"][name]
    return os.path.join(O.REF_DIR, "scenes", GOLDEN_JSON[name]), int(meta["n_tri"])


def scene_dir(kind: str) -> str:
    """Directory the reference must run in so that the scene's relative model paths resolve."""
    if kind == "dragon":
        return scene_cache_dir()
    from oracle import ct_oracle_py as O
    return os.path.join(O.REF_DIR, "scenes")


def load_host_scene(kind: str, refl):
    """The product's host scene for a workload: parsed by the product's own parser (dragon) or rebuilt from the
    flattened golden scene (the bundled scenes; tests prove both routes give the reference's triangles and BVH)."""
    import cobbletrace_b200 as ct
    from cobbletrace_b200 import host
    t0 = time.time()
    if kind == "dragon":
        path, _ = ensure_scene(kind)
        hs = host.HostScene.load(path, base_dir=scene_cache_dir())
    else:
        name = kind.split(":", 1)[1]
        meta = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["scenes"][name]
        hs = host.HostScene.from_flat(ct.load_ctscene(os.path.join(ROOT, "tests", "golden", meta["file"])).without_bvh())
    load_ms = (time.time() - t0) * 1e3
    if refl is not None:
        hs.set_reflection(refl)
    return hs, load_ms


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def ref_threads(height: int, cores: int) -> int:
    """numberOfThreads must divide H or the reference silently drops rows (raythread.cpp:576)."""
    return max(t for t in range(1, max(cores, 1) + 1) if height % t == 0)


# ---- clocks ----------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.mhz, self.reasons, self.max_mhz, self.err = index, False, [], set(), None, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self.stop_flag:
                self.mhz.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.005)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.mhz:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "error": self.err}
        return {"sm_mhz": float(np.median(self.mhz)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.mhz)}


DUMP_SAMPLE_PX = 1 << 22        # frames larger than 64 MB as float32 (dragon8k) are dumped as this many sampled pixels


def dump_frame(out_dir: str, frame: np.ndarray) -> None:
    """frame.npy: the read-back bitmap as float32 (its 0x00RRGGBB words are below 2^24, so the conversion is exact).
    Above 64 MB, a fixed sample of DUMP_SAMPLE_PX pixels (seed 0, in raster order) and their flat indices in
    frame_index.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    vals = frame.astype(np.float32)
    if vals.nbytes > 64 << 20:
        idx = np.sort(np.random.default_rng(0).choice(frame.size, DUMP_SAMPLE_PX, replace=False))
        np.save(os.path.join(out_dir, "frame_index.npy"), idx.astype(np.float64))
        vals = vals.reshape(-1)[idx]
    np.save(os.path.join(out_dir, "frame.npy"), vals)


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ---- reference arm / CPU baseline ----------------------------------------------------------------------------
def oracle_counts(fs, W, H, depth):
    """Reference-DFS ray and test counts for the frame (restatement; counters proven equal to oracle/_ref's in tests)."""
    from oracle import ct_oracle_py as O
    t0 = time.time()
    frame, _, ctr = O.OracleScene(fs).render(W, H, max_depth=depth, want_hits=False, by_kind=True)
    ctr["oracle_seconds"] = time.time() - t0
    from cobbletrace_b200.sceneio import frame_fnv1a
    ctr["frame_fnv1a"] = frame_fnv1a(frame)
    return ctr


def run_ref_cpu(scene_json, chdir, W, H, depth, refl, threads, frames, warmup, timeout=1500):
    from oracle import ct_oracle_py as O
    exe = os.path.join(O.REF_DIR, "ct_ref")
    cmd = [exe, "--scene", scene_json, "--chdir", chdir, "--width", str(W), "--height", str(H), "--depth", str(depth), "--threads", str(threads),
           "--time", str(frames), "--warmup", str(warmup)]
    if refl is not None:
        cmd += ["--force-reflection", repr(float(refl))]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=timeout).stdout
    return json.loads(out.strip().splitlines()[-1])


def cpu_baseline(workload, fs, counts_full, budget_s=25.0):
    """The reference's CPU renderer on this box's cores, on a bounded sample of the workload (rank 0, N = 1)."""
    from oracle import ct_oracle_py as O
    desc, kind, W, H, depth, refl = workload[:6]
    cores = host_cores()
    scene_path, _ = ensure_scene(kind)
    rays_full = counts_full["rays_primary"] + counts_full["rays_shadow"] + counts_full["rays_reflection"]
    if O.ref_available():
        # calibrate on a 1/16-area frame, then choose the largest sample that fits the budget (frame cost ~ pixels)
        w, h = W // 4, H // 4
        thr = ref_threads(h, cores)
        cal = run_ref_cpu(os.path.basename(scene_path), scene_dir(kind), w, h, depth, refl, thr, 1, 0)
        est_full = cal["best_ms"] * 16 / 1e3
        scale = 1
        while est_full / (scale * scale) > budget_s and scale < 8:
            scale *= 2
        w, h = W // scale, H // scale
        thr = ref_threads(h, cores)
        r = run_ref_cpu(os.path.basename(scene_path), scene_dir(kind), w, h, depth, refl, thr, 2, 0)
        rays = rays_full / (scale * scale)          # ray counts scale with the pixel count (same view, same scene)
        if scale > 1:
            c = oracle_counts(fs, w, h, depth)
            rays = c["rays_primary"] + c["rays_shadow"] + c["rays_reflection"]
        return {"value": rays / r["best_ms"] / 1e3, "unit": "Mrays/s", "cores": thr, "kind": "reference",
                "ms_per_frame": r["best_ms"], "host_cores": cores,
                "sample": f"{w}x{h} frame of the same scene/depth ({'full workload' if scale == 1 else f'1/{scale * scale} of the pixels'}), "
                          f"reference boss/worker with numberOfThreads={thr}, best of 2 frames, g++ -O2 -ffp-contract=off",
                "load_ms": r["load_ms"], "bvh_build_ms": r["build_ms"]}
    # no compiled reference on this box: time the plain-C restatement instead
    t0 = time.time()
    O.OracleScene(fs).render(W // 2, H // 2, max_depth=depth, want_hits=False, n_threads=cores)
    dt = time.time() - t0
    c = oracle_counts(fs, W // 2, H // 2, depth)
    rays = c["rays_primary"] + c["rays_shadow"] + c["rays_reflection"]
    return {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": f"{W // 2}x{H // 2} frame (1/4 of the pixels), oracle/ct_oracle.c with {cores} pthreads"}


def ref_counters(scene_json, chdir, W, H, depth, refl, threads, timeout=3000):
    """Ray / test counters of one frame from the compiled reference itself (oracle/_ref/ct_ref_count --counters)."""
    from oracle import ct_oracle_py as O
    cmd = [os.path.join(O.REF_DIR, "ct_ref_count"), "--scene", scene_json, "--chdir", chdir, "--width", str(W), "--height", str(H), "--depth", str(depth),
           "--threads", str(threads), "--counters"]
    if refl is not None:
        cmd += ["--force-reflection", repr(float(refl))]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=timeout).stdout
    return json.loads(out.strip().splitlines()[-1])


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.  Nothing of the
    product is loaded here: the scene file comes from the (pure Python) generator / the reference's own scene files, the
    frame times from oracle/_ref/ct_ref and the ray counts from oracle/_ref/ct_ref_count."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    from oracle import ct_oracle_py as O
    workload = WORKLOADS[args.workload]
    desc, kind, W, H, depth, refl = workload[:6]
    scene_path, n_tri = ensure_scene(kind)
    cores = host_cores()
    steps, warm = args.steps, args.warmup
    if O.ref_available():
        w, h = W // 4, H // 4
        cal = run_ref_cpu(os.path.basename(scene_path), scene_dir(kind), w, h, depth, refl, ref_threads(h, cores), 1, 0)
        est = cal["best_ms"] * 16 / 1e3 * (steps + warm + 1)
        scale = 1
        while est / (scale * scale) > 200 and scale < 8:
            scale *= 2
        w, h = W // scale, H // scale
        thr = ref_threads(h, cores)
        r = run_ref_cpu(os.path.basename(scene_path), scene_dir(kind), w, h, depth, refl, thr, steps, warm)
        ms = r["mean_ms"]
        c = ref_counters(os.path.basename(scene_path), scene_dir(kind), w, h, depth, refl, thr)
        n_nodes, n_lights = r["nodes"], r["lights"]
        kind_s, used = "reference", thr
        sample = (f"each step = one {w}x{h} frame ({'the full workload' if scale == 1 else f'1/{scale * scale} of the pixels'}) through the reference's "
                  f"boss/worker (AllocatePartitions/HandleUpdates/RayTracePartition), numberOfThreads={thr} of {cores} cores; "
                  "ray counts from the reference's own counters (ct_ref_count --counters)")
    else:
        # no compiled reference on this box: the plain-C restatement (needs the product's parser for the scene arrays)
        hs, _ = load_host_scene(kind, refl)
        fs = hs.to_flat(with_bvh=True)
        scale, w, h = 2, W // 2, H // 2
        osc = O.OracleScene(fs)
        for _ in range(warm):
            osc.render(w, h, max_depth=depth, want_hits=False, n_threads=cores)
        t0 = time.time()
        for _ in range(steps):
            osc.render(w, h, max_depth=depth, want_hits=False, n_threads=cores)
        ms = (time.time() - t0) / steps * 1e3
        c = oracle_counts(fs, w, h, depth)
        n_nodes, n_lights = fs.n_nodes, fs.n_lights
        kind_s, used = "port", cores
        sample = f"each step = one {w}x{h} frame (1/4 of the pixels) through oracle/ct_oracle.c with {cores} pthreads"
    rays = c["rays_primary"] + c["rays_shadow"] + c["rays_reflection"]
    value = rays / ms / 1e3
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64/f32 mixed (reference arithmetic)",
        "data": data_note(kind),
        "config": workload_config(args.workload, args.gpus, n_tri, n_nodes, n_lights),
        "sample": sample,
        "rays_per_step": {k: c[k] for k in ("rays_primary", "rays_shadow", "rays_reflection")},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": used, "kind": kind_s, "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- our arm -------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dragon4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tile-rows", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR/frame.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)
    # stdout carries exactly one line, the JSON (NCCL / torchrun banners go to stderr with everything else)
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from cobbletrace_b200 import api, build, host, multi
    import cobbletrace_b200 as ct

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cobbletrace_b200 has no CPU fallback")
    build.build_all()
    rank, local_rank, world = multi.init_distributed()
    if world != args.gpus:
        log(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    N = world
    dev = local_rank
    torch.cuda.set_device(dev)
    workload = WORKLOADS[args.workload]
    desc, kind, W, H, depth, refl = workload[:6]
    wflags = workload[6] if len(workload) > 6 else 0
    steps, warm = args.steps, max(args.warmup, 3)

    # ---- scene: generated, parsed and its BVH built ONCE per box (rank 0); the other ranks take a copy out of POSIX shared
    # memory (ct_host_scene_share / _attach).  The scene itself is replicated on every GPU (SURVEY 8e).
    shm_name = f"ct_bench_scene_{os.environ.get('MASTER_PORT', '0')}_{os.getuid()}"
    load_ms = bvh_ms = attach_ms = 0.0
    hs = None
    if rank == 0:
        scene_path, n_tri = ensure_scene(kind)
        hs, load_ms = load_host_scene(kind, refl)
        t0 = time.time(); n_nodes = hs.build_bvh(); bvh_ms = (time.time() - t0) * 1e3
        if N > 1:
            t0 = time.time(); hs.share(shm_name); attach_ms = (time.time() - t0) * 1e3
    if N > 1:
        dist.barrier()
        if rank != 0:
            t0 = time.time(); hs = host.HostScene.attach(shm_name); attach_ms = (time.time() - t0) * 1e3
            n_tri, n_nodes = hs.n_tri, hs.build_bvh()                      # (the BVH came with the copy: nothing is built)
        dist.barrier()
        if rank == 0:
            host.HostScene.unshare(shm_name)
    t0 = time.time()
    stream = torch.cuda.Stream(device=dev)
    cam_pos, cam_rot = hs.camera()
    n_lights = hs.n_lights
    # the reference-facing host path: the C++ boss (RayThread's boss half) uploads the scene arrays as they are
    boss = host.Boss(hs, W, H, devices=(dev,), max_depth=depth, tile_rows=args.tile_rows, flags=wflags)
    boss.set_stream(stream.cuda_stream)
    gpu = api.GpuRenderer(dev)                                              # the same device state, for the calls the boss does not wrap
    gpu.width, gpu.height = W, H
    shared = None
    if N > 1:
        # one process per GPU, one shared frame: chunks dealt / stolen from a cursor on GPU 0 over NVLink, pixels stored
        # straight into GPU 0's framebuffer (multi.SharedFrame / ct_gpu_render_shared)
        shared = multi.SharedFrame(gpu, root=0, stream=stream)
    upload_ms = (time.time() - t0) * 1e3
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{dev}")      # > 126 MB L2
    pinned = torch.zeros((H, W), dtype=torch.int32).pin_memory()
    bitmap = pinned.numpy().view(np.uint32)

    pinned2 = torch.zeros((H, W), dtype=torch.int32).pin_memory()
    bitmaps = [bitmap, pinned2.numpy().view(np.uint32)]

    def frame(to_host: bool, want_stats: bool = False, async_copy: int = -1):
        """One step.  Returns (stats or None, device_ms).  async_copy >= 0: the bitmap goes to the host through
        ct_gpu_readback_async into bitmaps[async_copy] (the copy overlaps the next frame) instead of ct_gpu_readback."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if N == 1:
            if to_host:
                boss.set_camera(cam_pos, 0.0, 0.0, 0.0)      # the per-frame input of the reference's boss (HandleUpdates :564-572)
            with torch.cuda.stream(stream):
                e0.record(stream)
                _, st = boss.render(bitmap if (to_host and async_copy < 0) else None, want_bitmap=False)
                e1.record(stream)
            if to_host and async_copy >= 0:
                gpu.readback_wait()                          # frame k - 1 has arrived ...
                gpu.readback_async(bitmaps[async_copy])      # ... frame k sets off, and travels while frame k + 1 renders
            stream.synchronize()
            return st, e0.elapsed_time(e1)
        shared.begin()                                       # rendezvous on the render stream (no cursor reset: two cursors alternate)
        if to_host:
            gpu.set_camera(cam_pos, cam_rot)                 # the camera is the per-frame input of every rank
        with torch.cuda.stream(stream):
            e0.record(stream)
            shared.render()
            e1.record(stream)
        shared.end()                                         # sync + barrier: the whole frame is in GPU 0's framebuffer
        if to_host and rank == 0:
            if async_copy >= 0:
                # snapshot in stream order BEFORE the next frame's rendezvous on the same stream: no rank can store into
                # the framebuffer until the snapshot is taken
                gpu.readback_wait()
                gpu.readback_async(bitmaps[async_copy])
            else:
                gpu.readback(bitmap)
        st = None
        if want_stats:
            st = gpu.counters(reset=True)
            st["tiles_total"] = 1
        return st, e0.elapsed_time(e1)

    def flush_l2():
        with torch.cuda.stream(stream):
            flush.fill_(1)
        stream.synchronize()

    def launches_so_far(reset=False):
        return gpu.kernel_launches(reset=reset) if N > 1 else 0

    def timed(to_host: bool, k: int, pipelined: bool = False):
        dev_ms, wall_ms, launches = [], [], 0
        launches_so_far(reset=True)
        for i in range(k):
            if not pipelined:
                flush_l2()
            t0 = time.perf_counter()
            st, ms = frame(to_host, async_copy=(i & 1) if pipelined else -1)
            wall_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(ms)
            if N == 1:
                launches += st["kernel_launches"]
        if pipelined and (N == 1 or rank == 0):
            gpu.readback_wait()
        launches += launches_so_far(reset=True)
        return np.array(dev_ms), np.array(wall_ms), launches

    for _ in range(warm):
        frame(False)
    if N > 1:
        gpu.counters(reset=True)
    st, _ = frame(False, want_stats=True)                    # the frame's ray counts (identical every frame)
    if N > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(physical_gpu_index(local_rank)); sampler.start()
    dev_ms, wall_ms, launches = timed(False, steps)
    torch.cuda.synchronize()
    if N > 1:
        dist.barrier()
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        dump_frame(args.dump_outputs, gpu.readback())          # GPU 0's framebuffer as the last timed step left it
    # end-to-end: host camera in, host bitmap out, wall clock -- one frame at a time (latency) ...
    for _ in range(2):
        frame(True)
    e2e_dev, e2e_wall, _ = timed(True, max(5, steps // 3))
    # ... and back to back with the copy of frame k overlapping the rendering of frame k + 1 (throughput of an interactive loop)
    n_pipe = max(8, steps // 2)
    frame(True, async_copy=0)
    if N > 1:
        dist.barrier()
    t0 = time.perf_counter()
    timed(True, n_pipe, pipelined=True)
    if N > 1:
        dist.barrier()
    pipe_ms = (time.perf_counter() - t0) * 1e3 / n_pipe
    frame(True)                                              # leaves the last frame in `bitmap` for the pixel check below
    # the same frames with every shadow ray traced (option shadow_reuse = 0): what the reuse of identical shadow rays is worth
    api.set_option("shadow_reuse", 0)
    for _ in range(2):
        frame(False)
    if N > 1:
        dist.barrier()
    noreuse_ms, _, _ = timed(False, max(5, steps // 4))
    api.set_option("shadow_reuse", 1)

    # ---- reduce over ranks: per-step max of the device time; sum of rays
    rays_vec = torch.tensor([st["rays_primary"], st["rays_shadow"], st["rays_reflection"], launches], dtype=torch.float64, device=f"cuda:{dev}")
    t_dev = torch.tensor(dev_ms, dtype=torch.float64, device=f"cuda:{dev}")
    t_e2e = torch.tensor(e2e_wall, dtype=torch.float64, device=f"cuda:{dev}")
    t_noreuse = torch.tensor(noreuse_ms, dtype=torch.float64, device=f"cuda:{dev}")
    t_once = torch.tensor([attach_ms + upload_ms if rank != 0 else 0.0], dtype=torch.float64, device=f"cuda:{dev}")
    if N > 1:
        dist.all_reduce(t_once, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays_vec, op=dist.ReduceOp.SUM)
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_noreuse, op=dist.ReduceOp.MAX)
    rays_primary, rays_shadow, rays_refl, total_launches = (int(x) for x in rays_vec.tolist())
    rays_total = rays_primary + rays_shadow + rays_refl
    ms_per_step = float(t_dev.mean())
    e2e_ms = float(t_e2e.mean())
    if rank != 0:
        shared.close(); boss.close()
        if N > 1:
            dist.barrier(); dist.destroy_process_group()
        return 0

    value = rays_total / ms_per_step / 1e3
    traced_px = rays_primary
    line = {
        "metric": metric_name(args.workload), "value": value, "unit": "Mrays/s", "n_gpus": N, "steps": steps, "warmup": warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64/f32 mixed (the reference's arithmetic, reproduced bit-exactly)",
        "data": data_note(kind),
        "config": workload_config(args.workload, N, n_tri, n_nodes, int(n_lights)),
        "method": {"timing": "CUDA events on the launching stream around each frame's kernels" + ("; max over ranks per step (pixels land in GPU 0's framebuffer inside those kernels)" if N > 1 else ""),
                   "tiles_per_frame": st["tiles_total"],
                   "parallelism": (f"{N} GPUs, one process each, scene replicated: 32-pixel chunks, 7/8 dealt round-robin and 1/8 stolen from one cursor on GPU 0 (atomics over NVLink), "
                                   "finished pixels stored straight into GPU 0's framebuffer (peer stores, CUDA IPC); no collective" if N > 1
                                   else "1 GPU; persistent warps steal 32-pixel chunks from a device-side cursor")},
        "ms_per_frame": ms_per_step,
        "rays_per_frame": {"primary": rays_primary, "shadow": rays_shadow, "reflection": rays_refl},
        "shadow_rays": {"counted": rays_shadow, "reused": None, "traced": None,
                        "note": ("rays are counted as the reference casts them (one shadow ray per light per shading point, raythread.cpp:304).  The reference's "
                                 "reflection rays have t = 0, so a reflection hit (tclosest = 0) puts the next shading point exactly on the previous one and "
                                 "ComputeLighting casts the same shadow rays again; this implementation answers those from the parent's verdicts ('reused') and "
                                 "traces the rest.  `without_shadow_reuse` is the same frame with option shadow_reuse = 0 (every ray traced)."),
                        "without_shadow_reuse": {"ms_per_step": float(t_noreuse.mean()), "value": rays_total / float(t_noreuse.mean()) / 1e3, "unit": "Mrays/s",
                                                 "steps": int(len(noreuse_ms))}},
        "mrays_per_s_by_kind": {"primary": rays_primary / ms_per_step / 1e3, "shadow": rays_shadow / ms_per_step / 1e3,
                                "reflection": rays_refl / ms_per_step / 1e3},
        "ms_per_step_min": float(t_dev.min()), "ms_per_step_max": float(t_dev.max()),
        "e2e": {"value": rays_total / e2e_ms / 1e3, "unit": "Mrays/s", "ms_per_frame": e2e_ms,
                "pipelined": {"value": rays_total / pipe_ms / 1e3, "unit": "Mrays/s", "ms_per_frame": pipe_ms, "frames": n_pipe,
                              "what": "the same loop back to back with ct_gpu_readback_async: frame k travels to the (pinned) host bitmap while frame k + 1 renders; wall clock over all frames, no L2 flush in between"},
                "h2d_bytes_per_step": 12 * 8, "d2h_bytes_per_step": int(traced_px) * 4,
                "what": ("ct_host_boss_set_camera (host doubles) + render + ct_gpu_readback into a pinned host bitmap, wall clock" if N == 1 else
                         "per frame: rendezvous (one-word all-reduce on the render stream), ct_gpu_set_camera on every rank, ct_gpu_render_shared, sync + barrier, "
                         "ct_gpu_readback of the whole frame on rank 0 into a pinned host bitmap; wall clock, max over ranks")},
        "gpu_launches": total_launches,
        "clocks": clocks,
        "one_time_ms": {"scene_parse": load_ms, "bvh_build": bvh_ms, "share_or_attach": attach_ms, "upload_and_alloc": upload_ms,
                        "other_ranks_max_total": float(t_once[0]),
                        "note": "rank 0's figures; at N > 1 only rank 0 parses and builds, the other ranks copy the scene out of shared memory (max over ranks below)"},
    }

    # ---- the pixels: the bitmap of the last end-to-end frame (read back from GPU 0, every rank's share in it) against the
    # frame the compiled, unmodified reference rendered for this workload (committed hash) -- at every N
    from cobbletrace_b200.sceneio import frame_fnv1a
    got_hash = frame_fnv1a(bitmap)
    want_hash, want_src = expected_frame(args.workload)
    line["frame_fnv1a"] = got_hash
    line["frame_check"] = {"reference_fnv1a": want_hash, "reference_source": want_src, "matches_reference": (got_hash == want_hash) if want_hash else None}
    frame_ok = (got_hash == want_hash) if want_hash else True

    # ---- roofline of the dominant kernel + CPU baseline (rank 0; only meaningful at N = 1)
    if N == 1 and wflags:
        boss.close()
        line["config"]["note"] = "sampling-mode stress workload: no roofline / CPU baseline (the reference's own supersampling is not reproducible)"
    elif N == 1:
        boss.close()
        fs = hs.to_flat(with_bvh=True)
        counts = oracle_counts(fs, W, H, depth)
        line["frame_check"]["oracle_fnv1a"] = counts["frame_fnv1a"]       # the live oracle render of the same inputs
        line["frame_check"]["matches_oracle"] = got_hash == counts["frame_fnv1a"]
        frame_ok = frame_ok and got_hash == counts["frame_fnv1a"]
        prof = api.GpuRenderer(dev).upload(fs, W, H, max_depth=depth, flags=api.CT_FLAG_STAGE_TIMING)
        per = {}
        for i in range(3 + 5):
            flush_l2()
            prof.render_tile()
            if i >= 3:
                for name, d, ms in prof.last_tile_stages():
                    per.setdefault(name, []).append(ms)
        n_frames = 5
        tot = {k: sum(v) / n_frames for k, v in per.items()}
        n_launch = {k: len(v) // n_frames for k, v in per.items()}
        prof.shutdown()
        # the GPU's OWN walk: box / triangle tests it actually performed for this frame (a counted frame, untimed)
        cnt = api.GpuRenderer(dev).upload(fs, W, H, max_depth=depth, flags=api.CT_FLAG_COUNT_TESTS)
        own = cnt.render_tile(counters=True)
        own_exact = cnt.filter_stats()
        line["shadow_rays"]["reused"] = cnt.reuse_stats()
        line["shadow_rays"]["traced"] = rays_shadow - line["shadow_rays"]["reused"]
        cnt.shutdown()
        alg = {   # algorithmic bytes per frame of each kernel type: 32 B per node visit + 48 B per triangle test of the
                  # REFERENCE's DFS on this frame, + 4 B per stored pixel (SURVEY 8d).  k_shadow owns the shadow rays
                  # (the rays it parks are finished by k_overflow, whose time is charged to it below)
            "primary": 32 * counts["box_tests_primary"] + 48 * counts["tri_tests_primary"] + 4 * traced_px,
            "shadow": 32 * counts["box_tests_shadow"] + 48 * counts["tri_tests_shadow"],
            "bounce": 32 * counts["box_tests_reflection"] + 48 * counts["tri_tests_reflection"],
        }
        tot_k = dict(tot)
        tot_k["primary"] = tot.get("primary", 0.0) + tot.get("primary_long", 0.0) + tot.get("primary_split", 0.0)   # (options primary_budget / primary_split)
        tot_k["shadow"] = tot.get("shadow", 0.0) + tot.get("overflow_shadow", 0.0)
        tot_k["bounce"] = tot.get("bounce", 0.0) + tot.get("overflow_bounce", 0.0)
        dominant = max(("primary", "shadow", "bounce"), key=lambda k: tot_k.get(k, 0.0))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = alg[dominant] / (tot_k[dominant] * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dominant)
        except Exception:
            pass
        frame_alg = sum(alg.values())
        # two yardsticks that do not saturate (the section-8d figure charges an any-hit walk with the reference's full
        # closest-hit DFS): (1) the same 32 B / 48 B per test, but for the tests THIS implementation performed;
        own_bytes = 32 * own["box_tests"] + 48 * own["tri_tests"] + 4 * traced_px
        own_walk = {"box_tests": own["box_tests"], "tri_tests": own["tri_tests"], "box_tests_fp64": own_exact[0], "tri_tests_fp64": own_exact[1],
                    "bytes": own_bytes, "achieved_GBps": own_bytes / (ms_per_step * 1e-3) / 1e9, "frac": own_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                    "vs_reference_dfs": {"box": own["box_tests"] / max(counts["box_tests"], 1), "tri": own["tri_tests"] / max(counts["tri_tests"], 1)},
                    "note": "32 B per box test + 48 B per triangle test the GPU itself performed (CT_FLAG_COUNT_TESTS frame) + 4 B per pixel, over the timed frame"}
        # (2) issue-slot utilisation: warp instructions per frame (ncu capture of the same workload, profiles/issue.json) over
        # the issue slots the kernels' measured time offers (SMs x 4 schedulers x SM clock)
        issue = None
        try:
            prof_issue = json.load(open(os.path.join(ROOT, "profiles", "issue.json")))[args.workload]
            sm_hz = (clocks.get("sm_mhz") or prof_issue.get("sm_mhz_at_capture") or 1965.0) * 1e6
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
            per_k = {}
            for k, v in prof_issue["warp_instructions_per_frame"].items():
                t_ms = tot.get(k)
                if t_ms:
                    per_k[k] = {"warp_instructions": v, "ms": t_ms, "issue_utilisation": v / (n_sm * 4 * sm_hz * t_ms * 1e-3)}
            all_inst = sum(prof_issue["warp_instructions_per_frame"].values())
            issue = {"per_kernel": per_k, "frame": {"warp_instructions": all_inst, "issue_utilisation": all_inst / (n_sm * 4 * sm_hz * ms_per_step * 1e-3)},
                     "lanes_per_instruction": prof_issue.get("lanes_per_instruction"), "source": prof_issue.get("source"),
                     "note": "warp instructions from the ncu capture (static, same workload and build), times measured live: 1.0 = every scheduler issues every cycle"}
        except Exception:
            pass
        line["roofline"] = {
            "bound": "hbm", "kernel": f"k_{dominant}", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
            "launches_per_frame": n_launch.get(dominant), "kernel_ms_per_frame": tot_k[dominant],
            "algorithmic_bytes_per_launch": alg[dominant] / max(n_launch.get(dominant, 1), 1),
            "kernel_share_of_step": {k: v / sum(tot.values()) for k, v in tot.items()},
            "whole_frame": {"algorithmic_bytes": frame_alg, "achieved_GBps": frame_alg / (ms_per_step * 1e-3) / 1e9,
                            "frac": frame_alg / (ms_per_step * 1e-3) / 1e9 / peak,
                            "bytes_per_ray": frame_alg / (counts["rays_primary"] + counts["rays_shadow"] + counts["rays_reflection"])},
            "reference_dfs_counts": {k: counts[k] for k in counts if k.startswith(("box_tests", "tri_tests"))},
            "own_walk": own_walk,
            "issue": issue,
            "note": ("achieved = algorithmic bytes of the REFERENCE's walk (32 B per box test + 48 B per triangle test of its closest-hit DFS, "
                     "SURVEY 8d) / kernel time: a throughput normalisation, not traffic.  The hot set (fp32 child pairs + fp32 triangles, 76 MB) is "
                     "L2-resident and a shadow ray needs fewer tests than the reference's full closest-hit walk, so the figure can exceed the HBM peak; "
                     "`traffic` is the measured DRAM bytes per launch (ncu, profiles/traffic.json).  The kernels are issue/latency bound: "
                     "profiles/r01_ncu_traversal_*_final.txt"),
        }
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(workload, fs, counts)
    else:
        shared.close(); boss.close()
    line["frame_matches_oracle"] = bool(frame_ok) if (want_hash or "matches_oracle" in line["frame_check"]) else None
    print(json.dumps(line), file=real_stdout, flush=True)
    if N > 1:
        dist.barrier(); dist.destroy_process_group()
    if not frame_ok:
        log(f"FRAME MISMATCH: read back {got_hash}, expected {line['frame_check']}")
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())
