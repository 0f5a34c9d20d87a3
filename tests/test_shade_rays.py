"""ct_gpu_shade_rays / GpuRenderer.shade_rays: TraceRay's colour for caller rays held in device memory.

Every colour is checked bit for bit against the oracle's own TraceRay (ct_oracle_trace_many, tests/shade_oracle.c around the pinned
oracle/ct_oracle.c) and, at full size, against the pixels a frame wrote for the camera's rays.  The oracle entry itself is pinned to
the golden frames of the compiled reference first."""
import contextlib
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api
from conftest import ROOT, case_scene, load_frames
from oracle import ct_oracle_py as O
from test_walk_limits import OPTION_NAMES, axis_rays, comb, gpu, ray_families, reverse_leaf_order, soup, spine, stack  # noqa: F401 (gpu: fixture)

CT_ERR_INVALID, CT_ERR_NO_SCENE, CT_ERR_LIMIT = -1, -4, -5
BATCH = 1 << 20                         # rays per batch (kShadeBatch in ct_gpu.cu)
GOLDEN_CASES = ["cube_160", "cube_rot_160", "cube_wide_200x120", "cube_tall_90x150", "import_160", "pc_big_96", "bunny_160",
                "bunny_refl_d2_160", "bunny_refl_d10_128", "bunny_odd_161x161"]
SETTINGS = {
    "default": {},
    "budget6": dict(traversal_budget=6),                                   # shadow / reflection rays parked for k_overflow
    "warp1": dict(traversal_budget=6, overflow_warp_budget=1),             # ... and handed on to k_overflow_huge
    "long1": dict(primary_budget=1),                                       # primary rays parked for k_primary_long
    "long6": dict(primary_budget=6),
    "split1": dict(primary_budget=1, primary_split=1),                     # ... for k_primary_split
    "split6": dict(primary_budget=6, primary_split=1),
    "reuse0": dict(shadow_reuse=0),                                        # every shadow ray traced, none taken from a parent
}


@contextlib.contextmanager
def options(**kw):
    try:
        for k, v in kw.items():
            api.set_option(k, v)
        yield
    finally:
        for k in OPTION_NAMES:
            api.set_option(k, 0)
        api.set_option("shadow_reuse", 1)


# ---- the oracle's TraceRay for caller rays -----------------------------------------------------------------------------------
_oracle = {}


def oracle_lib():
    """tests/shade_oracle.c compiled (into a temporary directory) with oracle/Makefile's flags for the restatement."""
    if "L" not in _oracle:
        out = os.path.join(tempfile.mkdtemp(prefix="ct_shade_oracle_"), "libct_shade_oracle.so")
        subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-std=c11",
                               "-I", os.path.join(ROOT, "oracle"), "-o", out, os.path.join(ROOT, "tests", "shade_oracle.c"), "-lm", "-lpthread"])
        L = C.CDLL(out)
        L.ct_oracle_trace_many.restype = None
        L.ct_oracle_trace_many.argtypes = [C.POINTER(O._Scene), C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _oracle["L"] = L
    return _oracle["L"]


def oracle_colors(fs, o, d, max_depth, osc=None):
    """ct_oracle_trace_many: TraceRay({o, d, 1e30f}, 1, FINF, max_depth) per ray, uint32."""
    osc = osc or O.OracleScene(fs)
    o = np.ascontiguousarray(o, np.float64).reshape(-1, 3); d = np.ascontiguousarray(d, np.float64).reshape(-1, 3)
    out = np.zeros(len(o), np.uint32)
    oracle_lib().ct_oracle_trace_many(C.byref(osc.c), len(o), o.ctypes.data, d.ctypes.data, int(max_depth), out.ctypes.data)
    return out


def canvas_rays(fs, H, x, y):
    """Primary rays through canvas points (x, y) with primary_ray_at's arithmetic (viewport {1, 1, 1}): a float32 quotient 1 / H, then
    float64 products and sums in CanvasToViewport * rotation's order."""
    s = np.float64(np.float32(1.0) / np.float32(H))
    vx, vy = np.asarray(x, np.float64) * s, np.asarray(y, np.float64) * s
    m = np.asarray(fs.cam_rot, np.float64).reshape(9)
    d = np.stack([vx * m[0] + vy * m[3] + 1.0 * m[6], vx * m[1] + vy * m[4] + 1.0 * m[7], vx * m[2] + vy * m[5] + 1.0 * m[8]], 1)
    o = np.broadcast_to(np.asarray(fs.cam_pos, np.float64), d.shape).copy()
    return o, d


def frame_pixels(W, H):
    """The pixels a full frame (render_tile's full range) traces and stores, scanline order: canvas (x, y) and framebuffer (row, col),
    plus the permutation into the frame's own slot order (8x4 pixel blocks)."""
    half = H // 2
    x_lo, n_x = -half, 2 * half                                   # the centred square (no CT_FLAG_WIDE)
    y0, y1 = max(-half, half - (H - 1)), min(-half + H, half + 1)
    Y, X = np.meshgrid(np.arange(y1 - 1, y0 - 1, -1), np.arange(x_lo, x_lo + n_x), indexing="ij")
    x, y = X.ravel(), Y.ravel()
    row, col = half - y, x + W // 2
    keep = (row >= 0) & (row < H) & (col >= 0) & (col < W)
    x, y, row, col = x[keep], y[keep], row[keep], col[keep]
    ix, iy, bx = x - x_lo, y - y0, (n_x + 7) // 8
    blocks = np.argsort(((iy // 4) * bx + ix // 8) * 32 + (iy % 4) * 8 + ix % 8, kind="stable")
    return x, y, row, col, blocks


# ---- 1. the oracle entry against the golden frames (CPU) ------------------------------------------------------------------------
@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_oracle_entry_reproduces_the_golden_frames(case, golden, scene_loader):
    fs, meta = case_scene(case, golden, scene_loader)
    g = load_frames(case)
    W, H = meta["width"], meta["height"]
    row, col = np.nonzero(g["found"] != 0xFFFFFFFF)          # the pixels the reference traced and stored
    o, d = canvas_rays(fs, H, col - W // 2, H // 2 - row)
    got = oracle_colors(fs, o, d, meta["depth"])
    bad = np.flatnonzero(got != g["frame"][row, col])
    assert bad.size == 0, f"{case}: {bad.size} of {got.size} pixels differ"


def test_frame_pixels_cover_what_the_golden_frames_traced(golden):
    for case in GOLDEN_CASES:
        meta = golden["frames"][case]
        W, H = meta["width"], meta["height"]
        _, _, row, col, blocks = frame_pixels(W, H)
        traced = np.zeros((H, W), bool)
        traced[row, col] = True
        assert np.array_equal(traced, load_frames(case)["found"] != 0xFFFFFFFF), case
        assert np.array_equal(np.sort(blocks), np.arange(len(row)))


# ---- 2. every ray against the oracle (GPU) --------------------------------------------------------------------------------------
def with_mirrors(fs, rng):
    """A soup in which a third of the triangles are perfect mirrors and a third reflect half."""
    import dataclasses
    refl = rng.choice(np.array([0.0, 0.5, 1.0], np.float32), fs.n_tri)
    return dataclasses.replace(fs, mat_reflection=refl)


def scene(name, scene_loader, rng):
    if name == "soup_mirrors":
        return with_mirrors(soup(rng, 500), rng)
    if name == "comb96":
        return comb(95, rng)
    if name == "spine":
        return spine(rng)
    if name == "reversed":
        return reverse_leaf_order(with_mirrors(soup(rng, 600), rng))
    if name == "bunny_refl":
        return scene_loader("scene_import_bunny").with_reflection(0.5)
    return scene_loader(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["scene_file_cube", "scene_import", "pc_big", "scene_import_bunny", "bunny_refl", "soup_mirrors", "comb96",
                                  "spine", "reversed"])
def test_every_ray_matches_the_oracle(name, scene_loader, gpu):
    import torch
    rng = np.random.default_rng(sum(map(ord, name)) + 11)
    fs = scene(name, scene_loader, rng)
    fam = ray_families(fs, rng, scale=0.25 if name in ("scene_import_bunny", "bunny_refl", "pc_big") else 0.6)
    if name in ("comb96", "spine"):
        fam.update(axis_rays(rng))
    o, d = stack(fam)
    reflective = bool((fs.mat_reflection > 0).any())
    depths = (0, 1, 2, 10) if reflective else (2,)
    osc = O.OracleScene(fs)
    ref = {k: oracle_colors(fs, o, d, k, osc) for k in depths}
    ref[None] = ref[depths[-1]]                                # the upload's depth below is the last one
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    small = fs.n_nodes + fs.n_tri <= 384                       # a tree this small parks at all only with a small traversal budget
    for setting, kw in SETTINGS.items():
        kw = dict(kw, traversal_budget=6) if small and "primary_budget" in kw else kw
        with options(**kw):
            gpu.upload(fs, 32, 32, max_depth=depths[-1])
            for k in depths + (None,):
                got = gpu.shade_rays(ot, dt, k).cpu().numpy().view(np.uint32)
                bad = np.flatnonzero(got != ref[k])
                assert bad.size == 0, (f"{name} {setting} max_depth {k}: {bad.size} of {got.size} rays differ, first ray {bad[0]}: "
                                       f"{got[bad[0]]:#08x} against {ref[k][bad[0]]:#08x}")


# ---- 3. the frame as the second oracle, at full size ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bench_dragon():
    """bench.py's dragon4k workload scene: the procedural stand-in, reflection forced to 0.5, the host BVH."""
    import bench
    hs, _ = bench.load_host_scene("dragon", bench.REFLECTION)
    return hs.to_flat(with_bvh=True)


def frame_and_colors(gpu, fs, W, H, depth):
    import torch
    gpu.upload(fs, W, H, max_depth=depth)
    gpu.render_tile()
    frame = gpu.readback()
    x, y, row, col, blocks = frame_pixels(W, H)
    o, d = canvas_rays(fs, H, x, y)
    ot, dt = (torch.from_numpy(a).to("cuda:0") for a in (o, d))
    return frame[row, col], ot, dt, blocks


def assert_pixels(got, want, what):
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} of {got.size} rays differ from the frame, first {bad[0]}: {got[bad[0]]:#08x} against {want[bad[0]]:#08x}"


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["dragon4k", "bunny1080"])
def test_camera_rays_equal_the_frame(workload, scene_loader, gpu, request):
    import torch
    if workload == "dragon4k":
        fs, W, H, depth = request.getfixturevalue("bench_dragon"), 3840, 2160, 2
    else:
        fs, W, H, depth = scene_loader("scene_import_bunny"), 1920, 1080, 10
    want, ot, dt, blocks = frame_and_colors(gpu, fs, W, H, depth)
    assert len(want) > BATCH                                    # several batches, and a partial last one
    got = gpu.shade_rays(ot, dt).cpu().numpy().view(np.uint32)
    assert_pixels(got, want, f"{workload} scanline order")
    p = torch.from_numpy(blocks).to("cuda:0")
    got = gpu.shade_rays(ot[p].contiguous(), dt[p].contiguous()).cpu().numpy().view(np.uint32)
    assert_pixels(got, want[blocks], f"{workload} 8x4 block order")


@pytest.mark.gpu
def test_batch_boundaries_on_a_small_scene(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_file_cube")
    W = H = 1024                                               # 1 047 552 traced pixels: just under one batch
    want, ot, dt, _ = frame_and_colors(gpu, fs, W, H, 10)
    rng = np.random.default_rng(12)
    for n in (BATCH - 1, BATCH, BATCH + 1):
        idx = rng.integers(0, len(want), n)
        p = torch.from_numpy(idx).to("cuda:0")
        got = gpu.shade_rays(ot[p].contiguous(), dt[p].contiguous()).cpu().numpy().view(np.uint32)
        assert_pixels(got, want[idx], f"n = {n}")


# ---- 4. order and batching ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_order_and_splitting_do_not_change_any_ray(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    rng = np.random.default_rng(13)
    o, d = stack(ray_families(fs, rng, scale=2.0))
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    for kw in ({}, dict(traversal_budget=6, primary_budget=1, primary_split=1)):
        with options(**kw):
            gpu.upload(fs, 32, 32, max_depth=3)
            base = gpu.shade_rays(ot, dt).cpu().numpy()
            for perm in (torch.randperm(len(o), generator=torch.Generator().manual_seed(5)), torch.arange(len(o) - 1, -1, -1)):
                p = perm.to("cuda:0")
                got = gpu.shade_rays(ot[p].contiguous(), dt[p].contiguous()).cpu().numpy()
                assert np.array_equal(got[np.argsort(perm.numpy())], base), f"permuted {kw}"
            k = len(o) // 3
            two = torch.cat([gpu.shade_rays(ot[:k], dt[:k]), gpu.shade_rays(ot[k:], dt[k:])]).cpu().numpy()
            assert np.array_equal(two, base), f"two calls {kw}"
            assert np.array_equal(gpu.shade_rays(o[7:8], d[7:8]), base[7:8].view(np.uint32))         # n = 1, numpy in and out
            assert gpu.shade_rays(ot[:0], dt[:0]).shape == (0,)                                     # n = 0


# ---- 5. streams, frames, counters, re-upload -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_colors_are_ordered_on_a_torch_side_stream(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_file_cube")
    rng = np.random.default_rng(14)
    o, d = stack(ray_families(fs, rng))
    ref = oracle_colors(fs, o, d, 10)
    gpu.upload(fs, 32, 32)
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = gpu.shade_rays(ot, dt)
        red = (c & 0xff).sum()                       # torch work on the same stream, no host synchronisation in between
        kept = c.clone()
    side.synchronize()
    assert int(red) == int((ref & 0xff).astype(np.int64).sum())
    assert np.array_equal(kept.cpu().numpy().view(np.uint32), ref)


@pytest.mark.gpu
def test_a_query_between_two_tiles_leaves_the_frame_alone(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    rng = np.random.default_rng(15)
    o, d = stack(ray_families(fs, rng, scale=0.3))
    ref = oracle_colors(fs, o, d, 3)
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    W = H = 96
    with options(traversal_budget=6, primary_budget=1):
        gpu.upload(fs, W, H, max_depth=3, flags=ct.CT_FLAG_COUNT_TESTS)
        gpu.render_tile()
        alone = gpu.readback()
        # queries count nothing: the frame counters, kernel launches, overflow and reuse statistics stay where the frame left them
        before = gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()
        gpu.shade_rays(ot, dt)
        assert (gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()) == before
        render = torch.cuda.Stream()
        render.wait_stream(torch.cuda.current_stream())
        gpu.set_stream(render.cuda_stream)
        y0, y1 = gpu.full_range()
        with torch.cuda.stream(render):
            gpu.render_tile(y0, (y0 + y1) // 2)
            got = gpu.shade_rays(ot, dt)
            gpu.render_tile((y0 + y1) // 2, y1)
        gpu.sync()
        gpu.set_stream(None)
        assert np.array_equal(got.cpu().numpy().view(np.uint32), ref)
        assert np.array_equal(gpu.readback(), alone)


@pytest.mark.gpu
def test_a_query_followed_at_once_by_a_new_upload(scene_loader, gpu):
    import torch
    fs = scene_loader("pc_big")                                 # 66 lights: three occlusion words per path
    rng = np.random.default_rng(16)
    o, d = stack(ray_families(fs, rng, scale=0.5))
    ref = oracle_colors(fs, o, d, 10)
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    with options(traversal_budget=6):
        gpu.upload(fs, 32, 32)
        got = gpu.shade_rays(ot, dt)                          # in flight ...
        gpu.upload(scene_loader("scene_file_cube"), 32, 32)    # ... while the scene it reads is replaced
    assert np.array_equal(got.cpu().numpy().view(np.uint32), ref)


# ---- 6. refusals, before anything is enqueued --------------------------------------------------------------------------------------
def query(n, o=None, d=None, color=None, max_depth=-1, size=None):
    q = api.ShadeQuery()
    q.struct_size = C.sizeof(api.ShadeQuery) if size is None else size
    q.n, q.max_depth = n, max_depth
    q.origins, q.directions, q.color = o, d, color
    return q


def rc(gpu, q):
    return gpu.L.ct_gpu_shade_rays(gpu.device, None if q is None else C.byref(q))


@pytest.mark.gpu
def test_refusals(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_file_cube")
    gpu.upload(fs, 32, 32)
    n = 64
    rng = np.random.default_rng(17)
    o, d = stack(ray_families(fs, rng, scale=0.1))
    o, d = np.ascontiguousarray(o[:n]), np.ascontiguousarray(d[:n])
    ot, dt = (torch.from_numpy(a).to("cuda:0") for a in (o, d))
    out = torch.zeros(n + 1, dtype=torch.int32, device="cuda:0")
    good = dict(o=ot.data_ptr(), d=dt.data_ptr(), color=out.data_ptr())
    pinned = torch.from_numpy(o).pin_memory()
    # every refusal with a canary: the sentinel in out[0..n] must survive (nothing was enqueued)
    out.fill_(-7)
    torch.cuda.synchronize()
    for bad in (dict(good, o=o.ctypes.data), dict(good, d=pinned.data_ptr()), dict(good, color=np.zeros(n, np.uint32).ctypes.data),
                dict(good, o=ot.data_ptr() + 4), dict(good, color=out.data_ptr() + 2), dict(good, o=None), dict(good, d=None),
                dict(good, color=None)):
        assert rc(gpu, query(n, **bad)) == CT_ERR_INVALID, bad
    assert rc(gpu, query(n, size=C.sizeof(api.ShadeQuery) - 8, **good)) == CT_ERR_INVALID
    assert rc(gpu, query(n, size=C.sizeof(api.RayQuery), **good)) == CT_ERR_INVALID
    assert rc(gpu, None) == CT_ERR_INVALID
    assert rc(gpu, query(1 << 31, **good)) == CT_ERR_LIMIT
    assert rc(gpu, query(n, max_depth=16, **good)) == CT_ERR_LIMIT
    if torch.cuda.device_count() > 1:
        assert rc(gpu, query(n, **dict(good, o=ot.to("cuda:1").data_ptr()))) == CT_ERR_INVALID
    torch.cuda.synchronize()
    assert bool((out == -7).all())
    # accepted: n = 0 with no arrays, max_depth 15 and < 0
    assert rc(gpu, query(0)) == 0
    assert rc(gpu, query(n, max_depth=15, **good)) == 0
    assert rc(gpu, query(n, max_depth=-5, **good)) == 0
    torch.cuda.synchronize()
    assert int(out[n]) == -7                                         # nothing written past n
    assert np.array_equal(out[:n].cpu().numpy().view(np.uint32), oracle_colors(fs, o, d, 10))
    for bad in (ot.float(), torch.zeros((n, 6), dtype=torch.float64, device="cuda:0")[:, ::2], ot.cpu(), ot[:, :2].contiguous()):
        with pytest.raises(ValueError):
            gpu.shade_rays(bad, dt)
    with pytest.raises(ValueError):
        gpu.shade_rays(ot, dt[:-1])
    with pytest.raises(api.CtError):
        gpu.shade_rays(ot, dt, 16)
    gpu.shutdown()
    assert rc(gpu, query(n, **good)) == CT_ERR_NO_SCENE
    assert rc(gpu, query(0)) == CT_ERR_NO_SCENE


def test_python_refuses_host_tensors_and_bad_depths():
    torch = pytest.importorskip("torch")
    if not os.path.exists(api.GPU_LIB):
        pytest.skip("libct_gpu.so not built")
    r = ct.GpuRenderer(0)
    o = torch.zeros((4, 3), dtype=torch.float64)
    for bad in (o, o.float(), o.numpy().tolist()):
        with pytest.raises(ValueError):
            r.shade_rays(bad, o)
    for depth in (1.5, "2", True, 1 << 40):
        with pytest.raises(ValueError):
            r.shade_rays(o, o, depth)
