"""ct_gpu_update_triangles / GpuRenderer.update_triangles: a loaded scene's triangles replaced from device memory, the reference's
tree rebuilt over them on the device, in place.

The result must be THE SAME SCENE as a fresh upload of the new triangles with CT_FLAG_BUILD_BVH and the scene's materials and lights:
every array ct_gpu_debug_scene_array exports, byte for byte.  Frames and ray / shade queries that follow must equal the oracle's on the
deformed scene, bit for bit.  What the update must keep (the caller's stream, camera, counters, launches, the previous frame) and the
refusals (each with the arrays and the frame unchanged) are checked one by one."""
import ctypes as C
import dataclasses
import time

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api, host, procedural
from cobbletrace_b200.sceneio import FlatScene
from oracle import ct_oracle_py as O

from conftest import load_fuzz_case
from test_device_bvh import GOLDEN_SCENES, comb_of_depth
from test_shade_rays import oracle_colors, options, with_mirrors
from test_trace_rays import assert_same, host_results, oracle_answers, KINDS
from test_walk_limits import _lights_and_camera, _materials, ray_families, reverse_leaf_order, stack

CT_ERR_INVALID, CT_ERR_NO_SCENE, CT_ERR_LIMIT = -1, -4, -5


@pytest.fixture
def gpu():
    r = ct.GpuRenderer(0)
    yield r
    r.shutdown()


def scene_arrays(r):
    return {k: r.debug_scene_array(k).tobytes() for k in api.SCENE_ARRAYS}


def laid_out(tri, stride):
    """Triangles at `stride` bytes, as GpuRenderer.upload lays them out (NaNs after the 9 doubles)."""
    tri = np.ascontiguousarray(tri, np.float64).reshape(-1, 9)
    if stride == 72:
        return tri
    wide = np.full((tri.shape[0], stride // 8), np.nan)
    wide[:, :9] = tri
    return wide


def update_abi(r, ptr, n, stride=72, size=None, stream=None):
    """ct_gpu_update_triangles with a hand-made descriptor; returns the status."""
    u = api.TriangleUpdate()
    u.struct_size = C.sizeof(api.TriangleUpdate) if size is None else size
    u.n_triangles, u.triangle_stride, u.triangles, u.stream = n, stride, ptr, stream
    return r.L.ct_gpu_update_triangles(r.device, C.byref(u))


def update_strided(r, tri, stride):
    import torch
    t = torch.from_numpy(laid_out(tri, stride)).to("cuda:0")
    rc = update_abi(r, t.data_ptr(), t.shape[0], stride)
    assert rc == 0, r.L.ct_gpu_last_error().decode()


def moved(fs, tri):
    """fs with new triangles and the reference's tree over them (what the oracle renders)."""
    return dataclasses.replace(fs, tri=np.ascontiguousarray(tri, np.float64).reshape(-1, 9), **O.build_bvh(tri))


def same_as_upload(r, fs, new_tri, what, W=16, H=16, stride=72, start_bvh=False, **kw):
    """Upload fs (its own tree, or built on the device), update it to new_tri, and compare with a fresh upload of new_tri."""
    r.upload(fs.without_bvh() if start_bvh else fs, W, H, triangle_stride=stride, build_bvh=start_bvh, **kw)
    update_strided(r, new_tri, stride)
    got = scene_arrays(r)
    r.upload(dataclasses.replace(fs, tri=np.asarray(new_tri, np.float64).reshape(-1, 9)).without_bvh(), W, H, triangle_stride=stride,
             build_bvh=True, **kw)
    want = scene_arrays(r)
    bad = [k for k in api.SCENE_ARRAYS if got[k] != want[k]]
    assert not bad, f"{what}: {bad} differ from a fresh upload"
    return np.frombuffer(want["summary"], api.SUMMARY_DT)[0]


def jitter(tri, rng, amount):
    scale = np.abs(tri).max() or 1.0
    return tri + rng.normal(size=tri.shape) * amount * scale


def tris_in_front(rng, n):
    c = rng.normal(size=(n, 3)) * 1.5 + np.array([0.0, 0.0, 6.0])
    a, b = rng.normal(size=(n, 3)) * 0.6, rng.normal(size=(n, 3)) * 0.6
    return np.concatenate([c - (a + b) / 3, c - (a + b) / 3 + a, c - (a + b) / 3 + b], 1)


def bare_scene(tri, rng, reflection=0.5):
    return FlatScene(tri=np.asarray(tri, np.float64), **_materials(rng, len(tri), reflection), **_lights_and_camera())


# ---- 1. the same scene as a fresh upload ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_same_scene_as_a_fresh_upload_golden(name, scene_loader, gpu):
    rng = np.random.default_rng(sum(map(ord, name)))
    fs = scene_loader(name)
    same_as_upload(gpu, fs, jitter(fs.tri, rng, 1e-3), name)
    same_as_upload(gpu, fs, jitter(fs.tri, rng, 3e-2), name + " (stride 96, device tree first)", stride=96, start_bvh=True)


@pytest.mark.gpu
def test_same_scene_as_a_fresh_upload_fuzz(gpu):
    rng = np.random.default_rng(31)
    for k in range(20):
        fs, _ = load_fuzz_case(f"{k:02d}")
        same_as_upload(gpu, fs, jitter(fs.tri, rng, 1e-2), f"fuzz_{k:02d}", stride=(72, 96, 120)[k % 3])


@pytest.mark.gpu
def test_same_scene_as_a_fresh_upload_dragon(tmp_path, gpu):
    scene, _ = procedural.write_dragon_standin(str(tmp_path))
    fs = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    s = same_as_upload(gpu, fs, jitter(fs.tri, np.random.default_rng(32), 1e-4), "dragon stand-in", W=64, H=64, max_depth=2)
    assert s["n_wide"] > 0 and s["can_overflow"] == 1


@pytest.mark.gpu
def test_a_host_tree_against_the_dfs_becomes_buildbvhs(scene_loader, gpu):
    fs = reverse_leaf_order(scene_loader("scene_import"))
    gpu.upload(fs, 16, 16)
    assert gpu.debug_scene_array("summary")["leaf_dfs_order"] == 0
    s = same_as_upload(gpu, fs, fs.tri, "scene_import, leaves in reverse DFS order")
    assert s["leaf_dfs_order"] == 1


# ---- 2. capacity transitions ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_leaf_root_and_soup_grow_and_shrink(gpu):
    rng = np.random.default_rng(33)
    n = 300
    same = np.tile(tris_in_front(rng, 1), (n, 1))                    # one leaf of n triangles: no pairs, no wide tree
    soup_a, soup_b = tris_in_front(rng, n), tris_in_front(rng, n)
    fs = bare_scene(same, rng)
    steps = (("leaf root -> soup (reallocated)", soup_a), ("soup -> leaf root (reused)", same), ("leaf root -> another soup", soup_b),
             ("soup -> soup", soup_a))
    want = {}
    for what, tri in steps:                                            # fresh uploads first: the update chain below runs uninterrupted
        gpu.upload(dataclasses.replace(fs, tri=tri).without_bvh(), 16, 16, build_bvh=True)
        want[what] = scene_arrays(gpu)
    gpu.upload(fs.without_bvh(), 16, 16, build_bvh=True)
    for what, tri in steps:
        update_strided(gpu, tri, 72)
        got = scene_arrays(gpu)
        assert (np.frombuffer(got["summary"], api.SUMMARY_DT)[0]["n_wide"] == 0) == (tri is same), what
        bad = [k for k in api.SCENE_ARRAYS if got[k] != want[what][k]]
        assert not bad, f"{what}: {bad} differ from a fresh upload"


def frames_match_oracle(r, fs, W, H, depth, what):
    r.render_tile()
    got = r.readback()
    want, _, _ = O.OracleScene(fs).render(W, H, max_depth=depth, want_hits=False)
    assert np.array_equal(got, want), f"{what}: {int((got != want).sum())} pixels differ"


@pytest.mark.gpu
@pytest.mark.parametrize("n, budget", [(190, 0), (4, 6)])
def test_can_overflow_turns_on(n, budget, gpu):
    """n identical triangles (a leaf root) cannot run past the visit budget; a soup of n can: the update allocates the parking
    buffers and pair_parent then, and the frames that follow park rays into them."""
    rng = np.random.default_rng(n)
    soup = tris_in_front(rng, n)
    fs = with_mirrors(bare_scene(np.tile(soup[:1], (n, 1)), rng), rng)
    W = H = 48
    with options(traversal_budget=budget, primary_budget=1):
        gpu.upload(fs.without_bvh(), W, H, max_depth=2, build_bvh=True)
        assert gpu.debug_scene_array("summary")["can_overflow"] == 0
        assert gpu.debug_scene_array("pair_parent").size == 0
        update_strided(gpu, soup, 72)
        got = scene_arrays(gpu)
        s = np.frombuffer(got["summary"], api.SUMMARY_DT)[0]
        assert s["can_overflow"] == 1 and len(got["pair_parent"]) == 4 * int(s["n_pairs"])
        frames_match_oracle(gpu, moved(fs, soup), W, H, 2, f"n = {n}")
        if budget:
            assert gpu.overflow_stats()[0] > 0                      # rays were parked into the buffers the update allocated
        gpu.upload(dataclasses.replace(fs, tri=soup).without_bvh(), W, H, max_depth=2, build_bvh=True)
        assert scene_arrays(gpu) == got


# ---- 3. frames and queries on a deforming mesh ------------------------------------------------------------------------------------
def deform(t0, step):
    """A seeded wave through the mesh, on the GPU (torch, current stream)."""
    import torch
    v = t0.view(-1, 3, 3)
    ext = (v.amax((0, 1)) - v.amin((0, 1))).clamp_min(1e-9)
    phase = (v - v.amin((0, 1))) / ext * 6.0 + 0.7 * step
    out = v + 0.02 * ext * torch.sin(phase[..., [1, 2, 0]])
    return out.reshape(-1, 9).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bunny", "mirror_soup"])
@pytest.mark.parametrize("depth", [0, 2])
def test_animation_matches_the_oracle(name, depth, scene_loader, gpu):
    import torch
    rng = np.random.default_rng(34 + depth)
    if name == "bunny":
        fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    else:
        fs = with_mirrors(bare_scene(tris_in_front(rng, 500), rng), rng)
        fs = host.HostScene.from_flat(fs).to_flat(with_bvh=True)
    W = H = 40
    gpu.upload(fs, W, H, max_depth=depth)
    t0 = torch.from_numpy(np.ascontiguousarray(fs.tri, np.float64)).to("cuda:0")
    for step in range(3):
        t = deform(t0, step)
        gpu.update_triangles(t)                                        # read in the current stream's order: no synchronisation
        cur = moved(fs, t.cpu().numpy())
        frames_match_oracle(gpu, cur, W, H, depth, f"{name} step {step}")
        o, d = stack(ray_families(cur, rng, scale=0.1))
        ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
        ref = oracle_answers(cur, o, d)
        for kind in KINDS:
            assert_same(host_results(gpu.trace_rays(ot, dt, kind)), ref[kind], f"{name} step {step} {kind}")
        got = gpu.shade_rays(ot, dt).cpu().numpy().view(np.uint32)
        want = oracle_colors(cur, o, d, depth)
        assert np.array_equal(got, want), f"{name} step {step}: {int((got != want).sum())} colours differ"


# ---- 4. what the update keeps -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_state_that_survives(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    W = H = 48
    rng = np.random.default_rng(35)
    gpu.upload(fs, W, H, max_depth=2, flags=ct.CT_FLAG_COUNT_TESTS)
    cam = np.asarray(fs.cam_pos, np.float64) + np.array([0.01, -0.02, 0.05])
    rot = O.camera_rotation(yaw=0.05, pitch=-0.03)
    gpu.set_camera(cam, rot)
    gpu.render_tile()
    before_frame = gpu.readback().copy()
    before = gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()
    side = torch.cuda.Stream()
    gpu.set_stream(side.cuda_stream)
    new = jitter(fs.tri, rng, 2e-3)
    gpu.update_triangles(new)
    assert (gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()) == before
    assert np.array_equal(gpu.readback(), before_frame)                # the previous frame until the next render
    # the library still renders on the caller's stream: ct_gpu_sync waits for work queued there
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
    t = time.perf_counter()
    gpu.sync()
    assert time.perf_counter() - t > 0.01
    gpu.render_tile()
    gpu.sync()
    gpu.set_stream(None)
    cur = dataclasses.replace(moved(fs, new), cam_pos=cam, cam_rot=np.asarray(rot, np.float64).reshape(9))
    want, _, _ = O.OracleScene(cur).render(W, H, max_depth=2, want_hits=False)
    assert np.array_equal(gpu.readback(), want)                        # the camera set before the update, the new triangles
    assert gpu.counters()["rays_primary"] > before[0]["rays_primary"]


# ---- 5. stream order ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_triangles_are_read_in_the_callers_stream_order(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import")
    new = jitter(fs.tri, np.random.default_rng(36), 5e-2)
    gpu.upload(fs, 16, 16)
    buf = torch.from_numpy(np.ascontiguousarray(fs.tri, np.float64)).to("cuda:0")
    src = torch.from_numpy(new).to("cuda:0")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)                                 # the triangles are written well after the call is made
        buf.copy_(src)
        gpu.update_triangles(buf)
    got = scene_arrays(gpu)
    gpu.upload(dataclasses.replace(fs, tri=new).without_bvh(), 16, 16, build_bvh=True)
    assert scene_arrays(gpu) == got


# ---- 6. refusals --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_change_nothing(gpu):
    import torch
    rng = np.random.default_rng(37)
    deep = comb_of_depth(97)
    fs = with_mirrors(bare_scene(tris_in_front(rng, len(deep)), rng), rng)
    W = H = 32
    gpu.upload(fs.without_bvh(), W, H, max_depth=2, build_bvh=True)
    gpu.render_tile()
    frame, arrays = gpu.readback().copy(), scene_arrays(gpu)
    n = fs.n_tri
    good = torch.from_numpy(jitter(fs.tri, rng, 1e-2)).to("cuda:0")
    wide = torch.zeros((n + 1, 9), dtype=torch.float64, device="cuda:0")
    host_tri = np.ascontiguousarray(fs.tri)
    pinned = torch.from_numpy(host_tri).pin_memory()
    cases = {
        "host pageable": dict(ptr=host_tri.ctypes.data, n=n),
        "host pinned": dict(ptr=pinned.data_ptr(), n=n),
        "misaligned": dict(ptr=good.data_ptr() + 4, n=n),
        "n + 1": dict(ptr=wide.data_ptr(), n=n + 1),
        "n - 1": dict(ptr=good.data_ptr(), n=n - 1),
        "stride 76": dict(ptr=good.data_ptr(), n=n, stride=76),
        "stride 64": dict(ptr=good.data_ptr(), n=n, stride=64),
        "struct_size": dict(ptr=good.data_ptr(), n=n, size=C.sizeof(api.TriangleUpdate) - 8),
        "NULL triangles": dict(ptr=None, n=n),
    }
    for what, kw in cases.items():
        assert update_abi(gpu, **kw) == CT_ERR_INVALID, what
    assert gpu.L.ct_gpu_update_triangles(0, None) == CT_ERR_INVALID
    d = torch.from_numpy(deep).to("cuda:0")
    assert update_abi(gpu, d.data_ptr(), n) == CT_ERR_LIMIT                # BuildBVH's tree over them is 97 deep
    assert scene_arrays(gpu) == arrays
    assert np.array_equal(gpu.readback(), frame)
    gpu.render_tile()
    assert np.array_equal(gpu.readback(), frame)                           # the previous triangles render as before
    for bad in (good.float(), good.cpu(), good[:-1], good.reshape(-1, 3), torch.zeros((n, 18), dtype=torch.float64, device="cuda:0")[:, ::2]):
        with pytest.raises(ValueError):
            gpu.update_triangles(bad)
    assert scene_arrays(gpu) == arrays
    gpu.update_triangles(good.view(n, 3, 3))                               # (n, 3, 3) is accepted
    gpu.shutdown()
    assert update_abi(gpu, good.data_ptr(), n) == CT_ERR_NO_SCENE


def test_python_refuses_what_it_cannot_read_in_place():
    torch = pytest.importorskip("torch")
    import os
    if not os.path.exists(api.GPU_LIB):
        pytest.skip("libct_gpu.so not built")
    r = ct.GpuRenderer(0)
    t = torch.zeros((4, 9), dtype=torch.float64)
    for bad in (t, t.float(), t.view(4, 3, 3), t.tolist(), None):
        with pytest.raises(ValueError):
            r.update_triangles(bad)
