"""Upload with the tree built on the device (CT_FLAG_BUILD_BVH) and the wide-tree collapse on the device.

An upload from bare triangles must build THE SAME SCENE as an upload of the host-built tree: every array ct_gpu_debug_scene_array
exports, byte for byte, and golden frames.  The wide tree (`wide`), now collapsed by a device kernel on both upload paths, is
compared with a restatement of the host loop it replaces, on caller trees too: garbage in unreachable slots, leaves out of DFS
order, the depth-96 comb, a leaf root.  Error paths: a tree passed with the flag, and a tree too deep to render, refused with
the previous scene still loaded."""
import dataclasses
import os

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api, host, procedural
from cobbletrace_b200.sceneio import FlatScene
from oracle import ct_oracle_py as O

from conftest import GOLD, load_frames, case_scene, load_fuzz_case
from test_walk_limits import comb, reverse_leaf_order, _lights_and_camera, _materials
from test_device_bvh import comb_of_depth, GOLDEN_SCENES

pytestmark = pytest.mark.gpu

K_WIDE_LEVELS = 2                       # CT_WIDE_LEVELS, the default build
K_WIDE = 1 << K_WIDE_LEVELS
WIDE_DT = np.dtype([("bmin", "<f4", 3), ("bmax", "<f4", 3), ("ref", "<u4"), ("cnt", "<u4")])


@pytest.fixture
def gpu():
    r = ct.GpuRenderer(0)
    yield r
    r.shutdown()


def scene_arrays(r):
    return {k: r.debug_scene_array(k).tobytes() for k in api.SCENE_ARRAYS}


def same_scene(gpu, fs, what, W=16, H=16, **kw):
    gpu.upload(fs, W, H, **kw)
    want = scene_arrays(gpu)
    gpu.upload(fs.without_bvh(), W, H, build_bvh=True, **kw)
    got = scene_arrays(gpu)
    bad = [k for k in api.SCENE_ARRAYS if got[k] != want[k]]
    assert not bad, f"{what}: {bad} differ"
    return want


def host_wide(fs):
    """The host loop ct_gpu_upload_scene ran before the collapse moved to the device: a queue of wide nodes, each holding
    K_WIDE_LEVELS levels of the tree below its interior node, children in DFS order, interior children numbered as queued."""
    left, count, first = fs.node_left, fs.node_count, fs.node_first
    if count[0] != 0:
        return np.zeros(0, WIDE_DT)
    root_of, out = [0], []
    w = 0
    while w < len(root_of):
        cur = [int(left[root_of[w]]), int(left[root_of[w]]) + 1]
        for _ in range(1, K_WIDE_LEVELS):
            nxt = []
            for c in cur:
                nxt += [c] if count[c] != 0 else [int(left[c]), int(left[c]) + 1]
            cur = nxt
        rec = np.zeros(K_WIDE, WIDE_DT)
        for i in range(K_WIDE):
            if i >= len(cur):
                rec[i] = ((1e30,) * 3, (-1e30,) * 3, 0xFFFFFFFF, 0)
                continue
            c = cur[i]
            ref = int(first[c]) if count[c] else len(root_of)
            if not count[c]:
                root_of.append(c)
            rec[i] = (fs.node_min[c].astype(np.float32), fs.node_max[c].astype(np.float32), ref, int(count[c]))
        out.append(rec)
        w += 1
    return np.concatenate(out)


def check_wide(gpu, fs, what):
    gpu.upload(fs, 16, 16)
    got = gpu.debug_scene_array("wide")
    want = host_wide(fs)
    assert got.tobytes() == want.tobytes(), f"{what}: wide tree differs ({got.size // 32} / {want.size} entries)"
    assert int(gpu.debug_scene_array("summary")["n_wide"]) * K_WIDE == want.size


def scene_from_triangles(tri, rng, reflection=0.5):
    return FlatScene(tri=tri, **_materials(rng, tri.shape[0], reflection), **_lights_and_camera((0.5, 0.0, -2.0)))


# ---- the same scene from both upload paths ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_flag_upload_builds_the_same_scene_golden(name, scene_loader, gpu):
    same_scene(gpu, scene_loader(name), name)
    same_scene(gpu, scene_loader(name), name + " (stride 96)", triangle_stride=96)


def test_flag_upload_builds_the_same_scene_fuzz(gpu):
    for k in range(20):
        fs, _ = load_fuzz_case(f"{k:02d}")
        same_scene(gpu, fs, f"fuzz_{k:02d}", triangle_stride=(72, 96, 120)[k % 3])


def test_flag_upload_builds_the_same_scene_dragon(tmp_path, gpu):
    scene, _ = procedural.write_dragon_standin(str(tmp_path))
    fs = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    s = same_scene(gpu, fs, "dragon stand-in")
    assert np.frombuffer(s["summary"], api.SUMMARY_DT)[0]["n_wide"] > 0


@pytest.mark.parametrize("case", ["cube_160", "import_160", "pc_big_96", "bunny_refl_d2_160"])
def test_flag_upload_renders_golden_frames(case, golden, scene_loader, gpu):
    fs, meta = case_scene(case, golden, scene_loader)
    gpu.upload(fs.without_bvh(), meta["width"], meta["height"], max_depth=meta["depth"], build_bvh=True)
    gpu.render_tile()
    want = load_frames(case)["frame"]
    got = np.zeros_like(want)
    gpu.readback(got)
    assert np.array_equal(got, want), f"{case}: {int((got != want).sum())} pixels differ"


def test_flag_upload_renders_a_supersampled_golden_frame(golden, scene_loader, gpu):
    m = golden["frames_supersampling"]["bunny_refl_d2_80x60"]
    fs = scene_loader(m["scene"]).with_reflection(m["force_reflection"])
    gpu.upload(fs.without_bvh(), m["width"], m["height"], max_depth=m["depth"], flags=ct.CT_FLAG_SUPERSAMPLING, build_bvh=True)
    gpu.render_tile()
    want = np.load(os.path.join(GOLD, "frames_ss_bunny_refl_d2_80x60.npz"))["frame"]
    got = np.zeros_like(want)
    gpu.readback(got)
    assert np.array_equal(got, want)


# ---- the wide collapse on the device, caller trees ------------------------------------------------------------------------------
def test_device_wide_collapse_on_caller_trees(scene_loader, gpu):
    rng = np.random.default_rng(21)
    for name in GOLDEN_SCENES:
        check_wide(gpu, scene_loader(name), name)
    fs = scene_loader("scene_import")
    check_wide(gpu, reverse_leaf_order(fs), "scene_import, leaves in reverse DFS order")
    garbage = np.frombuffer(rng.bytes(64 * 9), api.NODE_DT)                   # slots the tree never reaches may hold anything
    g = dataclasses.replace(fs, node_min=np.concatenate([fs.node_min, garbage["min"]]), node_max=np.concatenate([fs.node_max, garbage["max"]]),
                            node_left=np.concatenate([fs.node_left, garbage["left"]]), node_first=np.concatenate([fs.node_first, garbage["first"]]),
                            node_count=np.concatenate([fs.node_count, garbage["count"]]))
    check_wide(gpu, g, "scene_import with garbage in unreachable slots")
    check_wide(gpu, comb(95, rng), "comb of depth 96")
    leaf = scene_from_triangles(np.array([[0.0, 0, 1, 1, 0, 1, 0, 1, 1], [0.0, 0, 2, 1, 0, 2, 0, 1, 2]]), rng)
    leaf = dataclasses.replace(leaf, **O.build_bvh(leaf.tri))
    assert leaf.node_count[0] == 2
    check_wide(gpu, leaf, "leaf root")
    assert gpu.debug_scene_array("wide").size == 0
    same_scene(gpu, leaf, "leaf root")


# ---- error paths --------------------------------------------------------------------------------------------------------------
def test_flag_with_a_tree_is_refused(scene_loader, gpu):
    fs = scene_loader("scene_file_cube")
    with pytest.raises(ct.CtError) as e:
        gpu.upload(fs, 16, 16, flags=api.CT_FLAG_BUILD_BVH)                  # the flag, and a tree
    assert e.value.code == -1
    with pytest.raises(ValueError):
        gpu.upload(fs.without_bvh(), 16, 16)                                 # neither: as before


def test_too_deep_a_built_tree_is_refused_and_the_scene_stays(gpu):
    rng = np.random.default_rng(5)
    ok = scene_from_triangles(comb_of_depth(96), rng)
    gpu.upload(ok, 48, 48, max_depth=3, build_bvh=True)
    assert int(gpu.debug_scene_array("summary")["depth"]) == 96
    gpu.render_tile()
    before = gpu.readback().copy()
    arrays = scene_arrays(gpu)
    deep = scene_from_triangles(comb_of_depth(97), rng)
    with pytest.raises(ct.CtError) as e:
        gpu.upload(deep, 48, 48, max_depth=3, build_bvh=True)
    assert e.value.code == -5
    assert scene_arrays(gpu) == arrays
    gpu.render_tile()
    assert np.array_equal(gpu.readback(), before)
    want, _, _ = O.OracleScene(dataclasses.replace(ok, **O.build_bvh(ok.tri))).render(48, 48, max_depth=3, want_hits=False)
    assert np.array_equal(before, want)
