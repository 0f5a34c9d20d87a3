"""ct_gpu_update_scene / GpuRenderer.update_scene: a loaded scene's triangles (of any count), materials and lights replaced from device
memory.

After every update the device must hold THE SAME SCENE as a fresh upload with CT_FLAG_BUILD_BVH of the resulting triangles, materials
and lights: every array ct_gpu_debug_scene_array exports (api.SCENE_STATE: the tree's arrays, the light records and what the path state
was sized from), byte for byte.  Chains of updates run on one renderer, so that allocations reused after a shrink and a grow are tested
too.  Frames and ray / shade queries that follow must equal the oracle's on the edited scene, bit for bit.  What the update must keep and
the refusals (each with the state and the frame unchanged) are checked one by one."""
import ctypes as C
import dataclasses
import os
import shutil
import subprocess
import time

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api, host, procedural
from cobbletrace_b200.sceneio import LT_AMBIENT, LT_DIRECTIONAL, LT_POINT
from oracle import ct_oracle_py as O

from conftest import load_fuzz_case
from test_device_bvh import GOLDEN_SCENES, comb_of_depth
from test_gpu_parity import assert_same as assert_frame_and_hits
from test_shade_rays import SETTINGS, options, oracle_colors
from test_trace_rays import KINDS, assert_same, host_results, oracle_answers
from test_update_triangles import bare_scene, frames_match_oracle, jitter, laid_out, tris_in_front
from test_walk_limits import ray_families, stack

CT_ERR_INVALID, CT_ERR_NO_DEVICE, CT_ERR_NO_SCENE, CT_ERR_LIMIT = -1, -2, -4, -5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def gpu():
    r = ct.GpuRenderer(0)
    yield r
    r.shutdown()


# ---- scenes and their parts -----------------------------------------------------------------------------------------------------
def state(r):
    return {k: r.debug_scene_array(k).tobytes() for k in api.SCENE_STATE}


def path_state(r):
    return r.debug_scene_array("path_state")


def materials_of(fs):
    m = np.zeros(fs.n_tri, api.MAT_DT)
    m["color"], m["specular"], m["reflection"] = fs.mat_color, fs.mat_specular, fs.mat_reflection
    return m


def lights_of(fs):
    lt = np.zeros(fs.n_lights, api.LIGHT_DT)
    lt["type"], lt["intensity"], lt["pos"], lt["dir"] = fs.light_type, fs.light_intensity, fs.light_pos, fs.light_dir
    return lt


SHADOW_DT = np.dtype([("type", "<i4"), ("index", "<u4"), ("v", "<f8", 3)])      # the device's shadow-light record


def shadow_lights_of(fs):
    """The lights ComputeLighting casts shadow rays to, in file order: every light but the ambient ones (raythread.cpp:284-286), towards
    a point light's position (:288) or along any other light's direction (:293)."""
    keep = np.flatnonzero(np.asarray(fs.light_type) != LT_AMBIENT)
    out = np.zeros(len(keep), SHADOW_DT)
    out["type"], out["index"] = np.asarray(fs.light_type)[keep], keep
    point = (np.asarray(fs.light_type)[keep] == LT_POINT)[:, None]
    out["v"] = np.where(point, np.reshape(fs.light_pos, (-1, 3))[keep], np.reshape(fs.light_dir, (-1, 3))[keep])
    return out


def as_tensors(fs, part):
    """The (color, specular, reflection) / (type, intensity, pos, dir) tuple update_scene takes, on cuda:0."""
    import torch
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to("cuda:0")
    if part == "materials":
        return (t(fs.mat_color, np.uint32).to(torch.int64), t(fs.mat_specular, np.int32), t(fs.mat_reflection, np.float32))
    return (t(fs.light_type, np.int32), t(fs.light_intensity, np.float32), t(np.reshape(fs.light_pos, (-1, 3)), np.float64),
            t(np.reshape(fs.light_dir, (-1, 3)), np.float64))


def random_lights(rng, n, n_shadow=None):
    """n lights in front of the camera, n_shadow of them point or directional (all of them when None), the rest ambient, shuffled."""
    n_shadow = n if n_shadow is None else n_shadow
    types = np.array([LT_AMBIENT] * (n - n_shadow) + list(rng.choice([LT_POINT, LT_DIRECTIONAL], n_shadow)), np.int32)
    rng.shuffle(types)
    pos = rng.normal(size=(n, 3)) * 4.0 + np.array([0.0, 0.0, -2.0])
    return dict(light_type=types, light_intensity=rng.uniform(0.01, 1.5 / max(n, 1), n).astype(np.float32),
                light_pos=pos.reshape(-1, 3), light_dir=rng.normal(size=(n, 3)).reshape(-1, 3))


def random_materials(rng, n, reflective):
    refl = rng.choice(np.array([0.0, 0.5, 1.0, -0.25], np.float32), n) if reflective else np.where(rng.random(n) < 0.5, 0.0, -1.0).astype(np.float32)
    return dict(mat_color=rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32),
                mat_specular=rng.choice(np.array([-1, 0, 10, 500], np.int32), n), mat_reflection=refl)


def edit(fs, **kw):
    return dataclasses.replace(fs, **kw).without_bvh()


def apply(r, fs, parts, numpy=False, stride=72):
    """update_scene with the given parts of fs (torch tensors, or numpy record arrays); stride != 72 goes through the ABI."""
    import torch
    if stride != 72:
        tri = torch.from_numpy(laid_out(fs.tri, stride)).to("cuda:0")
        m = torch.from_numpy(materials_of(fs).view(np.uint8)).to("cuda:0")
        lt = torch.from_numpy(lights_of(fs).view(np.uint8)).to("cuda:0")
        rc = update_abi(r, what=7, n=fs.n_tri, stride=stride, tri=tri.data_ptr(), mat=m.data_ptr(), n_lights=fs.n_lights,
                        lights=lt.data_ptr() if fs.n_lights else None)
        assert rc == 0, r.L.ct_gpu_last_error().decode()
        r.n_tri = fs.n_tri
        return
    kw = {}
    if "triangles" in parts:
        kw["triangles"] = fs.tri if numpy else torch.from_numpy(np.ascontiguousarray(fs.tri, np.float64)).to("cuda:0")
    if "materials" in parts:
        kw["materials"] = materials_of(fs) if numpy else as_tensors(fs, "materials")
    if "lights" in parts:
        kw["lights"] = lights_of(fs) if numpy else as_tensors(fs, "lights")
    r.update_scene(**kw)


def update_abi(r, what, n=0, stride=72, tri=None, mat=None, n_lights=0, lights=None, stream=None, size=None):
    """ct_gpu_update_scene with a hand-made descriptor; returns the status."""
    u = api.SceneUpdate()
    u.struct_size = C.sizeof(api.SceneUpdate) if size is None else size
    u.what, u.n_triangles, u.triangle_stride, u.n_lights = what, n, stride, n_lights
    u.triangles, u.materials, u.lights, u.stream = tri, mat, lights, stream
    return r.L.ct_gpu_update_scene(r.device, C.byref(u))


ALL = ("triangles", "materials", "lights")


def chain(r, start, steps, W=16, H=16, stride=72, start_bvh=True, **kw):
    """Fresh uploads of every step's scene first; then ONE renderer uploads `start` and applies the steps in turn, each compared with
    its fresh upload.  steps: (what, scene, parts).  Returns the path states."""
    want = []
    for what, fs, parts in steps:
        r.upload(fs.without_bvh(), W, H, triangle_stride=stride, build_bvh=True, **kw)
        want.append(state(r))
    r.upload(start.without_bvh() if start_bvh else start, W, H, triangle_stride=stride, build_bvh=start_bvh, **kw)
    out = []
    for k, (what, fs, parts) in enumerate(steps):
        apply(r, fs, parts, numpy=k % 2 == 1, stride=stride)
        got = state(r)
        bad = [n for n in api.SCENE_STATE if got[n] != want[k][n]]
        assert not bad, f"step {k} ({what}): {bad} differ from a fresh upload"
        assert got["lights"] == lights_of(fs).tobytes() and got["shadow_lights"] == shadow_lights_of(fs).tobytes(), what
        out.append(np.frombuffer(got["path_state"], api.PATH_DT)[0])
    return out


def soup_scene(rng, n, reflective=True, n_lights=3):
    return edit(bare_scene(tris_in_front(rng, n), rng), **random_materials(rng, n, reflective), **random_lights(rng, n_lights))


# ---- 1. the same scene as a fresh upload ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("depth", [0, 2, 10])
def test_material_edits_change_the_path_depth(depth, gpu):
    rng = np.random.default_rng(40 + depth)
    fs = soup_scene(rng, 300, reflective=False)
    nan = random_materials(rng, 300, False)
    nan["mat_reflection"][17] = np.nan                                     # a NaN reflection recurses as the reference does
    steps = [("reflective", edit(fs, **random_materials(rng, 300, True)), ("materials",)),
             ("none reflective", edit(fs, **random_materials(rng, 300, False)), ("materials",)),
             ("one NaN", edit(fs, **nan), ("materials",)),
             ("none again", edit(fs, **random_materials(rng, 300, False)), ("materials",))]
    got = chain(gpu, fs, steps, max_depth=depth)
    assert [int(s["any_reflective"]) for s in got] == [1, 0, 1, 0]
    assert [int(s["levels"]) for s in got] == [depth + 1, 1, depth + 1, 1]


@pytest.mark.gpu
def test_light_edits_change_the_occlusion_words(gpu):
    rng = np.random.default_rng(41)
    fs = soup_scene(rng, 400, n_lights=3)
    counts = [(0, 0), (1, 0), (66, 40), (33, 10), (3, 2)]                 # (lights, of them casting shadows)
    steps = [(f"{n} lights", edit(fs, **random_lights(rng, n, k)), ("lights",)) for n, k in counts]
    got = chain(gpu, fs, steps, max_depth=2)
    assert [int(s["occ_words"]) for s in got] == [1, 1, 3, 2, 1]
    assert [int(s["n_shadow_lights"]) for s in got] == [k for _, k in counts]
    assert [int(s["any_leaves"]) for s in got] == [12, 12, 8, 12, 12]
    # the option "any_leaves" keeps its upload-time value
    with options(any_leaves=5):
        gpu.upload(fs.without_bvh(), 16, 16, build_bvh=True)
    apply(gpu, steps[2][1], ("lights",))
    assert int(path_state(gpu)["any_leaves"]) == 5


@pytest.mark.gpu
def test_count_changes(gpu):
    rng = np.random.default_rng(42)
    fs = soup_scene(rng, 300)
    sizes = [800, 100, 1, 2, 500, 300]                                     # grow, shrink, a single triangle (a leaf root), grow again
    steps = []
    for k, n in enumerate(sizes):
        parts = ("triangles", "materials") if k % 2 else ALL
        nxt = edit(fs, tri=tris_in_front(rng, n), **random_materials(rng, n, k % 3 != 2),
                   **(random_lights(rng, 1 + 20 * k) if "lights" in parts else {}))
        steps.append((f"{n} triangles", nxt, parts))
        fs = nxt
    got = chain(gpu, soup_scene(rng, 300), steps, max_depth=2)
    assert [int(s["n_triangles"]) for s in got] == sizes
    assert gpu.debug_scene_array("summary")["root_cnt"] == 0


@pytest.mark.gpu
def test_fuzz_scenes_swapped_into_each_other(gpu):
    scenes = [load_fuzz_case(f"{k:02d}")[0] for k in range(20)]
    for stride in (72, 96, 120):
        steps = [(f"fuzz_{k:02d} stride {stride}", fs, ALL) for k, fs in enumerate(scenes[1:] + scenes[:1], 1)]
        chain(gpu, scenes[0], steps, stride=stride, start_bvh=stride != 72, max_depth=2)


@pytest.mark.gpu
def test_golden_scenes_swapped_into_each_other(scene_loader, gpu):
    scenes = [scene_loader(n) for n in GOLDEN_SCENES]
    steps = [(n, fs, ALL) for n, fs in zip(GOLDEN_SCENES[1:] + GOLDEN_SCENES[:1], scenes[1:] + scenes[:1])]
    chain(gpu, scenes[0], steps, W=32, H=32, start_bvh=False, max_depth=3)


@pytest.mark.gpu
def test_dragon_into_a_soup_and_back(tmp_path, gpu):
    rng = np.random.default_rng(43)
    path, _ = procedural.write_dragon_standin(str(tmp_path))
    dragon = host.HostScene.load(path, base_dir=str(tmp_path)).to_flat(with_bvh=True).with_reflection(0.5)
    small = soup_scene(rng, 60)                                            # 119 nodes + 60 triangles: no walk can be parked
    steps = [("soup", small, ALL), ("dragon", dragon, ALL), ("soup, materials and lights", edit(small, **random_lights(rng, 40)), ALL)]
    got = chain(gpu, dragon, steps, W=64, H=64, start_bvh=False, max_depth=2)
    assert [int(s["ovf_cap"]) > 0 for s in got] == [False, True, False]


# ---- 2. a seeded sequence of random edits on one renderer --------------------------------------------------------------------------
@pytest.mark.gpu
def test_random_edit_sequence(gpu):
    rng = np.random.default_rng(44)
    fs = start = soup_scene(rng, 200)
    steps = []
    for k in range(30):
        parts = [ALL, ("triangles", "materials"), ("materials",), ("lights",), ("materials", "lights"), ("triangles",)][rng.integers(6)]
        n = int(rng.choice([1, 5, 60, 200, 700])) if "materials" in parts and "triangles" in parts else fs.n_tri
        kw = {}
        if "triangles" in parts:
            kw["tri"] = tris_in_front(rng, n) if n != fs.n_tri else jitter(fs.tri, rng, 0.05)
        if "materials" in parts:
            kw.update(random_materials(rng, n, rng.random() < 0.6))
        if "lights" in parts:
            kw.update(random_lights(rng, int(rng.choice([0, 1, 3, 17, 40, 70])), None))
            kw["light_type"][rng.random(len(kw["light_type"])) < 0.2] = LT_AMBIENT
        fs = edit(fs, **kw)
        steps.append((f"{'+'.join(parts)} -> {n} triangles, {fs.n_lights} lights", fs, parts))
    chain(gpu, start, steps, W=24, H=24, max_depth=3)


# ---- 3. frames and queries on the edited scene ------------------------------------------------------------------------------------
def check_everything(r, fs, W, H, depth, what):
    import torch
    frames_match_oracle(r, fs, W, H, depth, what)
    o, d = stack(ray_families(fs, np.random.default_rng(45), scale=0.3))
    ot, dt = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0") for a in (o, d))
    ref = oracle_answers(fs, o, d)
    for kind in KINDS:
        assert_same(host_results(r.trace_rays(ot, dt, kind)), ref[kind], f"{what} {kind}")
    got = r.shade_rays(ot, dt).cpu().numpy().view(np.uint32)
    want = oracle_colors(fs, o, d, depth)
    assert np.array_equal(got, want), f"{what}: {int((got != want).sum())} colours differ"


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [0, 1, 2])
def test_frames_and_queries_match_the_oracle(depth, gpu):
    rng = np.random.default_rng(46 + depth)
    start = host.HostScene.from_flat(soup_scene(rng, 250, reflective=False)).to_flat(with_bvh=True)
    mirrors = dataclasses.replace(start, **random_materials(rng, 250, True))
    lit = dataclasses.replace(mirrors, **random_lights(rng, 66, 40))
    grown = bare_scene(tris_in_front(rng, 420), rng)
    grown = host.HostScene.from_flat(dataclasses.replace(grown, **random_materials(rng, 420, True), **random_lights(rng, 5),
                                                         cam_pos=start.cam_pos, cam_rot=start.cam_rot)).to_flat(with_bvh=True)
    steps = [("materials", mirrors, ("materials",)), ("66 lights", lit, ("lights",)), ("all three", grown, ALL)]
    W = H = 32
    for setting, kw in SETTINGS.items():
        kw = dict(kw, traversal_budget=6) if "primary_budget" in kw else kw      # a tree this small parks only with a small budget
        with options(**kw):
            gpu.upload(start, W, H, max_depth=depth)
            for what, fs, parts in steps:
                apply(gpu, fs, parts)
                check_everything(gpu, fs, W, H, depth, f"depth {depth} {setting} {what}")


# ---- 4. what the update keeps ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_state_that_survives(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    W = H = 48
    rng = np.random.default_rng(47)
    gpu.upload(fs, W, H, max_depth=2, flags=ct.CT_FLAG_COUNT_TESTS)
    cam = np.asarray(fs.cam_pos, np.float64) + np.array([0.01, -0.02, 0.05])
    rot = O.camera_rotation(yaw=0.05, pitch=-0.03)
    gpu.set_camera(cam, rot)
    gpu.render_tile()
    before_frame = gpu.readback().copy()
    before = gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()
    side = torch.cuda.Stream()
    gpu.set_stream(side.cuda_stream)
    n = fs.n_tri + 37
    new = host.HostScene.from_flat(edit(fs, tri=np.concatenate([fs.tri, jitter(fs.tri[:37], rng, 1e-2)]), **random_materials(rng, n, True),
                                        **random_lights(rng, 7))).to_flat(with_bvh=True)
    apply(gpu, new, ALL)
    assert (gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats(), gpu.kernel_launches()) == before
    assert np.array_equal(gpu.readback(), before_frame)                # the previous frame until the next render
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
    t = time.perf_counter()
    gpu.sync()                                                         # the library still renders on the caller's stream
    assert time.perf_counter() - t > 0.01
    gpu.render_tile()
    gpu.sync()
    gpu.set_stream(None)
    cur = dataclasses.replace(new, cam_pos=cam, cam_rot=np.asarray(rot, np.float64).reshape(9))
    want, _, _ = O.OracleScene(cur).render(W, H, max_depth=2, want_hits=False)
    assert np.array_equal(gpu.readback(), want)                        # the camera set before the update, the new scene
    assert gpu.counters()["rays_primary"] > before[0]["rays_primary"]


@pytest.mark.gpu
def test_kept_hits_and_a_shared_frame_after_an_update(scene_loader, gpu):
    rng = np.random.default_rng(48)
    fs = scene_loader("scene_import")
    W = H = 40
    gpu.upload(fs, W, H, max_depth=2, flags=ct.CT_FLAG_KEEP_HITS)
    gpu.share_attach(gpu.share_export())                               # self-attach: the shared-frame path on one device
    gpu.render_shared()
    n = fs.n_tri * 2
    new = host.HostScene.from_flat(edit(fs, tri=np.concatenate([fs.tri, jitter(fs.tri, rng, 3e-2)]), **random_materials(rng, n, True),
                                        **random_lights(rng, 4))).to_flat(with_bvh=True)
    apply(gpu, new, ALL)
    oframe, ohits, _ = O.OracleScene(new).render(W, H, max_depth=2)
    gpu.render_shared()
    gpu.sync()
    assert_frame_and_hits(gpu, oframe, ohits, "shared frame after an update")
    gpu.share_attach(None)
    gpu.render_tile()
    assert_frame_and_hits(gpu, oframe, ohits, "frame after an update")


# ---- 5. stream order -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_inputs_are_read_in_the_callers_stream_order(scene_loader, gpu):
    import torch
    rng = np.random.default_rng(49)
    fs = scene_loader("scene_import")
    n = fs.n_tri + 5
    new = edit(fs, tri=np.concatenate([jitter(fs.tri, rng, 5e-2), tris_in_front(rng, 5)]), **random_materials(rng, n, True),
               **random_lights(rng, 40, 20))
    gpu.upload(fs, 16, 16, max_depth=2)
    srcs = [torch.from_numpy(np.ascontiguousarray(new.tri)).to("cuda:0")] + list(as_tensors(new, "materials")) + list(as_tensors(new, "lights"))
    bufs = [torch.zeros_like(s) for s in srcs]
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)                                 # the inputs are written well after the call is made
        for b, s in zip(bufs, srcs):
            b.copy_(s)
        gpu.update_scene(triangles=bufs[0], materials=tuple(bufs[1:4]), lights=tuple(bufs[4:]))
    got = state(gpu)
    gpu.upload(new, 16, 16, max_depth=2, build_bvh=True)
    assert state(gpu) == got


# ---- 6. refusals -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_change_nothing(gpu):
    import torch
    rng = np.random.default_rng(50)
    deep = comb_of_depth(97)
    fs = soup_scene(rng, 300)
    W = H = 32
    gpu.upload(fs, W, H, max_depth=2, build_bvh=True)
    gpu.render_tile()
    frame, before = gpu.readback().copy(), state(gpu)
    n = fs.n_tri
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")
    tri, tri2 = cuda(jitter(fs.tri, rng, 1e-2)), cuda(tris_in_front(rng, n + 1))
    mat, mat2 = cuda(materials_of(fs).view(np.uint8)), cuda(np.resize(materials_of(fs), n + 1).view(np.uint8))
    lit = cuda(lights_of(fs).view(np.uint8))
    host_tri, host_mat = np.ascontiguousarray(fs.tri), materials_of(fs)
    pinned = torch.from_numpy(host_tri).pin_memory()
    T, M, L = api.CT_UPDATE_TRIANGLES, api.CT_UPDATE_MATERIALS, api.CT_UPDATE_LIGHTS
    good = dict(n=n, tri=tri.data_ptr(), mat=mat.data_ptr(), n_lights=fs.n_lights, lights=lit.data_ptr())
    invalid = {
        "struct_size": dict(good, what=7, size=C.sizeof(api.SceneUpdate) - 8),
        "what = 0": dict(good, what=0),
        "unknown bit": dict(good, what=7 | 8),
        "host triangles": dict(good, what=T, tri=host_tri.ctypes.data),
        "pinned triangles": dict(good, what=T, tri=pinned.data_ptr()),
        "host materials": dict(good, what=M, mat=host_mat.ctypes.data),
        "misaligned triangles": dict(good, what=T, tri=tri.data_ptr() + 4),
        "misaligned materials": dict(good, what=M, mat=mat.data_ptr() + 2),
        "misaligned lights": dict(good, what=L, lights=lit.data_ptr() + 4),
        "stride 76": dict(good, what=T, stride=76),
        "stride 64": dict(good, what=T, stride=64),
        "no triangles": dict(good, what=T | M, n=0),
        "NULL triangles": dict(good, what=T, tri=None),
        "NULL materials": dict(good, what=M, mat=None),
        "new count without materials": dict(good, what=T | L, n=n + 1, tri=tri2.data_ptr()),
        "materials alone, new count": dict(good, what=M, n=n + 1, mat=mat2.data_ptr()),
        "lights > 0, NULL": dict(good, what=L, lights=None),
    }
    for what, kw in invalid.items():
        assert update_abi(gpu, **kw) == CT_ERR_INVALID, what
    assert gpu.L.ct_gpu_update_scene(0, None) == CT_ERR_INVALID
    assert update_abi(gpu, **dict(good, what=T | M, n=1 << 31)) == CT_ERR_LIMIT
    d = cuda(deep)
    m_deep = cuda(np.resize(materials_of(fs), len(deep)).view(np.uint8))
    assert update_abi(gpu, **dict(good, what=7, n=len(deep), tri=d.data_ptr(), mat=m_deep.data_ptr())) == CT_ERR_LIMIT   # 97 deep
    assert state(gpu) == before
    assert np.array_equal(gpu.readback(), frame)
    gpu.render_tile()
    assert np.array_equal(gpu.readback(), frame)                           # the previous scene renders as before
    for kw in malformed(torch, n):
        with pytest.raises(ValueError):
            gpu.update_scene(**kw)
    assert state(gpu) == before
    gpu.shutdown()
    assert update_abi(gpu, **dict(good, what=7)) == CT_ERR_NO_SCENE


def malformed(torch, n, device="cuda:0"):
    """update_scene arguments that must raise ValueError (n: the loaded scene's triangle count)."""
    z = lambda *s, dt=torch.float64: torch.zeros(s, dtype=dt, device=device)
    tri = z(n, 9)
    mats = (z(n, dt=torch.int64), z(n, dt=torch.int32), z(n, dt=torch.float32))
    lts = (z(3, dt=torch.int32), z(3, dt=torch.float32), z(3, 3), z(3, 3))
    return [
        {},
        dict(triangles=tri.float()), dict(triangles=tri.cpu()), dict(triangles=z(n, 18)[:, ::2]), dict(triangles=tri.reshape(-1, 3)),
        dict(triangles=z(n + 1, 9)),                                       # a new count without new materials
        dict(triangles=z(0, 9), materials=tuple(a[:0] for a in mats)),
        dict(materials=tuple(a[:-1] for a in mats)),                       # materials alone keep the count
        dict(triangles=tri, materials=tuple(a[:-1] for a in mats)),
        dict(materials=mats[:2]), dict(materials=(mats[0].float(),) + mats[1:]), dict(materials=(mats[0],) + (mats[1].long(), mats[2])),
        dict(materials=(mats[0].cpu(),) + mats[1:]), dict(materials=(mats[0][:-1],) + mats[1:]), dict(materials=mats[0]),
        dict(materials=np.zeros(n, np.float64)), dict(materials=np.zeros((n, 1), api.MAT_DT)),
        dict(lights=lts[:3]), dict(lights=(lts[0].float(),) + lts[1:]), dict(lights=lts[:2] + (z(3, 2), lts[3])),
        dict(lights=lts[:3] + (z(4, 3),)), dict(lights=lts[:2] + (lts[2].float(), lts[3])), dict(lights=(lts[0].cpu(),) + lts[1:]),
        dict(lights=np.zeros(3, api.MAT_DT)), dict(lights=[1, 2, 3, 4]),
    ]


# ---- CPU: the ABI's layouts and the Python checks ---------------------------------------------------------------------------------
def test_ctypes_layouts_match_the_header(tmp_path):
    """SceneUpdate and PathSummary against sizeof / offsetof of the C99 header."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ct_gpu.h"\n'
                   "#define F(T, f) printf(#T \" \" #f \" %zu\\n\", offsetof(T, f))\n"
                   "int main(void) {\n"
                   '    printf("ct_scene_update size %zu\\n", sizeof(ct_scene_update));\n'
                   '    printf("ct_path_summary size %zu\\n", sizeof(ct_path_summary));\n'
                   + "".join(f"    F(ct_scene_update, {f});\n" for f, _ in api.SceneUpdate._fields_)
                   + "".join(f"    F(ct_path_summary, {f});\n" for f, _ in api.PathSummary._fields_)
                   + '    printf("mask %d %d %d\\n", CT_UPDATE_TRIANGLES, CT_UPDATE_MATERIALS, CT_UPDATE_LIGHTS);\n'
                   "    return 0;\n}\n")
    exe = str(tmp_path / "layout")
    subprocess.run([shutil.which("cc") or "cc", "-std=c99", "-Wall", "-Wextra", "-Werror", str(src), "-I", os.path.join(ROOT, "include"),
                    "-o", exe], check=True)
    lines = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines()
    assert lines[-1].split()[1:] == [str(api.CT_UPDATE_TRIANGLES), str(api.CT_UPDATE_MATERIALS), str(api.CT_UPDATE_LIGHTS)]
    out = dict((" ".join(l.split()[:2]), int(l.split()[2])) for l in lines[:-1])
    for T, cls in (("ct_scene_update", api.SceneUpdate), ("ct_path_summary", api.PathSummary)):
        assert out[f"{T} size"] == C.sizeof(cls), T
        for f, _ in cls._fields_:
            assert out[f"{T} {f}"] == getattr(cls, f).offset, f"{T}.{f}"
    assert C.sizeof(api.PathSummary) == api.PATH_DT.itemsize
    assert set(api.SCENE_STATE) == set(api.SCENE_ARRAYS) | {"lights", "shadow_lights", "path_state"}


def test_tensors_pack_into_the_librarys_records():
    """The records update_scene packs from tensors equal the ct_material / ct_light records of the numpy arrays (torch on the CPU)."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(51)
    fs = edit(bare_scene(tris_in_front(rng, 9), rng), **random_materials(rng, 9, True), **random_lights(rng, 5, 3))
    fs.mat_color[:3] = [0, 0x80000000, 0xFFFFFFFF]
    fs.mat_reflection[3] = np.nan
    cpu = torch.device("cpu")
    r = ct.GpuRenderer.__new__(ct.GpuRenderer)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt))
    want = materials_of(fs).view(np.uint8)
    for color in (t(fs.mat_color, np.int64), t(fs.mat_color, np.uint32)):
        got, n = r._device_materials((color, t(fs.mat_specular, np.int32), t(fs.mat_reflection, np.float32)), cpu)
        assert n == 9 and np.array_equal(got.numpy().view(np.uint8).ravel(), want), color.dtype
    for k in (5, 0):
        lt = dataclasses.replace(fs, **{f: getattr(fs, f)[:k] for f in ("light_type", "light_intensity", "light_pos", "light_dir")})
        parts = (t(lt.light_type, np.int64), t(lt.light_intensity, np.float32), t(lt.light_pos, np.float64), t(lt.light_dir, np.float64))
        got, n = r._device_lights(parts, cpu)
        assert n == k and np.array_equal(got.numpy().ravel(), lights_of(lt).view(np.uint8))


class _NoCalls:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name}) for a malformed argument")


def test_python_refuses_malformed_arguments_without_calling_the_library():
    torch = pytest.importorskip("torch")
    if not os.path.exists(api.GPU_LIB):
        pytest.skip("libct_gpu.so not built")
    r = ct.GpuRenderer(0)
    r.n_tri = 4
    r.L = _NoCalls()
    cpu = [dict(triangles=torch.zeros((4, 9), dtype=torch.float64)), dict(triangles=[[0.0] * 9] * 4), dict(materials=None, lights=None),
           dict(materials=(torch.zeros(4, dtype=torch.int64), torch.zeros(4, dtype=torch.int32), torch.zeros(4))),
           dict(lights=(torch.zeros(1, dtype=torch.int32), torch.zeros(1), torch.zeros((1, 3), dtype=torch.float64),
                        torch.zeros((1, 3), dtype=torch.float64))),
           dict(materials=np.zeros(4, np.float64)), dict(materials=np.zeros((4, 1), api.MAT_DT)), dict(lights=np.zeros(2, api.MAT_DT)),
           dict(materials="red"), dict(lights=(1, 2, 3, 4))]
    cases = cpu + (malformed(torch, 4) if torch.cuda.is_available() else [])
    for kw in cases:
        with pytest.raises(ValueError):
            r.update_scene(**kw)


def test_no_device_is_refused_by_the_entry_point():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = ct.GpuRenderer(0)
    assert update_abi(r, what=api.CT_UPDATE_LIGHTS) == CT_ERR_NO_DEVICE
    assert update_abi(r, what=0) == CT_ERR_INVALID                         # refused before the device is looked for
