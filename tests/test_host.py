"""Host side (libct_host.so): scene ingest, BVH build, camera matrix -- against reference-derived goldens,
and, when oracle/_ref is present, against the compiled reference run live on the same files."""
import math
import os

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import host, procedural
from oracle import ct_oracle_py as O

SCENES = ["scene_file_cube", "scene_import", "pc_big", "scene_import_bunny"]
REF_SCENES = os.path.join(O.REF_DIR, "scenes")
need_ref = pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref not built (needs the reference's sources: CT_REFERENCE_SRC)")


@pytest.mark.parametrize("name", SCENES)
def test_bvh_builder_is_bit_identical_to_reference(name, golden, scene_loader):
    fs = scene_loader(name)
    rebuilt = host.HostScene.from_flat(fs.without_bvh()).to_flat(with_bvh=True)
    assert rebuilt.bvh_digest() == golden["scenes"][name]["bvh_sha256"]
    assert rebuilt.n_nodes == golden["scenes"][name]["n_nodes"]


@need_ref
@pytest.mark.parametrize("name", SCENES)
def test_scene_loader_is_bit_identical_to_reference_parser(name, golden):
    hs = host.HostScene.load(os.path.join(REF_SCENES, name + ".json"), base_dir=REF_SCENES)
    fs = hs.to_flat(with_bvh=True)
    meta = golden["scenes"][name]
    assert fs.n_tri == meta["n_tri"] and fs.n_lights == meta["n_lights"]
    assert fs.geometry_digest() == meta["geometry_sha256"]
    assert fs.bvh_digest() == meta["bvh_sha256"]


def test_camera_rotation_float_semantics(golden):
    step = math.pi / 4 / 4
    for keys, g in golden["camera"].items():
        yaw = pitch = roll = np.float32(0)
        for k in keys:
            if k == "y": yaw = np.float32(np.float64(yaw) + step)
            if k == "p": pitch = np.float32(np.float64(pitch) + step)
            if k == "r": roll = np.float32(np.float64(roll) + step)
        assert np.array_equal(host.camera_rotation(yaw, pitch, roll), np.array(g["rot"])), keys
    ident = host.camera_rotation(0, 0, 0)
    assert np.array_equal(ident, np.array([1, 0, 0, 0, 1, 0, 0, 0, 1.0])) and np.signbit(ident[6])   # [2][0] = -0.0


SMALL_SCENE = """{
  "objects":[
    {"type": "sphere", "center": [0, 0, 6], "radius": 1.5, "color": [1, 2, 3], "specular": 10, "reflection": 0.5},
    {"type": "triangle", "p1": [0.1, 1e-1, -2.5e1], "p2": [-100, -100, 5], "p3": [100.25, -100, 5],
     "color": [255, 0.9, 300], "specular": -1, "reflection": 0.3333}
  ],
  "lights":[ {"type": "ambient", "intensity": 0.2}, {"type": "point", "intensity": 0.6, "position": [2, 1, 0]},
             {"type": "directional", "intensity": 0.2, "direction": [1, 4, 4]} ],
  "camera":{ "position": [0, 0.5, -3] },
  "settings":{ "numberOfThreads": 4, "subsampling": false, "wireframe": false, "supersampling": true }
}"""


def test_parser_number_and_colour_semantics(tmp_path):
    p = tmp_path / "s.json"
    p.write_text(SMALL_SCENE)
    hs = host.HostScene.load(str(p))
    fs = hs.to_flat(with_bvh=True)
    assert hs.n_tri == 1 and hs.n_spheres == 1 and fs.n_lights == 3
    f32 = np.float32
    # GetNumber accumulates in fp32 digit by digit (fileBuffer.cpp:160-207): 0.1 -> float(1/10), 1e-1 -> float(1 * pow(10,-1))
    assert fs.tri[0, 0] == np.float64(f32(1) / f32(10))
    assert fs.tri[0, 1] == np.float64(f32(np.float64(f32(1)) * 10.0 ** -1))
    assert fs.tri[0, 2] == -25.0 and fs.tri[0, 6] == 100.25
    # colour: double -> uint8 truncation, 300 wraps to 44, packed 0x00BBGGRR (scenefile.cpp:74, color.h:77)
    assert fs.mat_color[0] == ((300 & 0xFF) << 16) | (0 << 8) | 255
    assert fs.mat_specular[0] == -1 and fs.mat_reflection[0] == f32(0.3333)
    assert list(fs.light_type) == [ct.sceneio.LT_AMBIENT, ct.sceneio.LT_POINT, ct.sceneio.LT_DIRECTIONAL]
    assert hs.settings() == dict(numberOfThreads=4, subsampling=False, wireframe=False, supersampling=True)
    assert hs.render_flags() == ct.api.CT_FLAG_SUPERSAMPLING
    both = tmp_path / "both.json"
    both.write_text(SMALL_SCENE.replace('"subsampling": false', '"subsampling": true'))
    assert host.HostScene.load(str(both)).render_flags() == ct.api.CT_FLAG_SUPERSAMPLING | ct.api.CT_FLAG_SUBSAMPLING
    plain = tmp_path / "plain.json"
    plain.write_text(SMALL_SCENE.replace('"supersampling": true', '"supersampling": false'))
    assert host.HostScene.load(str(plain)).render_flags() == 0
    assert np.array_equal(fs.cam_pos, [0, 0.5, -3])


@pytest.mark.parametrize("bad,msg", [
    ('{"objects":[{"type":"cone"}]}', "unknown object type"),
    ('{"lights":[{"type":"ambient","colour":1}]}', "unknown light key"),
    ('{"settings":{"wireFrame": true}}', "unknown settings key"),       # utils/trisphere.json trips the reference's assert here
    ('{"camera":{"position":[0,0]}}', "expected"),
    ('{"objects":[{"type":"triangle","p1":[0,0,0],"p2":[1,0,0],"p3":[0,1,0]}]', "expected"),
])
def test_parser_reports_errors_instead_of_asserting(tmp_path, bad, msg):
    p = tmp_path / "bad.json"
    p.write_text(bad)
    with pytest.raises(RuntimeError) as e:
        host.HostScene.load(str(p))
    assert msg in str(e.value)


def test_missing_model_file_is_an_error(tmp_path):
    p = tmp_path / "s.json"
    p.write_text('{"objects":[{"type":"import","filename":"models/nope.ply","format":"ply","scale":[1,1,1]}]}')
    with pytest.raises(RuntimeError) as e:
        host.HostScene.load(str(p), base_dir=str(tmp_path))
    assert "cannot open" in str(e.value)


def test_procedural_standin_small(tmp_path):
    parts = procedural.small_standin_parts(3)
    scene, n = procedural.write_dragon_standin(str(tmp_path), parts=parts, name="mini")
    hs = host.HostScene.load(scene, base_dir=str(tmp_path))
    fs = hs.to_flat(with_bvh=True)
    assert fs.n_tri == n == sum(8 * 4 ** d for d, _, _ in parts)
    # the BVH restatement in the oracle agrees with the product builder on a scene neither has seen before
    b = O.build_bvh(fs.tri)
    assert all(np.array_equal(v, getattr(fs, k)) for k, v in b.items())
    # every vertex lies on its sphere (model units, before the import transform): check triangle count and closedness only
    v, f = procedural.octasphere(3)
    assert f.shape[0] == 8 * 4 ** 3 and v.shape[0] == f.shape[0] // 2 + 2
    assert np.allclose(np.linalg.norm(v, axis=1), 1.0)


@need_ref
def test_procedural_standin_parses_identically_in_reference(tmp_path):
    parts = procedural.small_standin_parts(4)
    scene, n = procedural.write_dragon_standin(str(tmp_path), parts=parts, name="mini")
    dump = str(tmp_path / "ref.ctscene")
    O.run_ref(os.path.basename(scene), chdir=str(tmp_path), width=16, height=16, threads=1, dump_scene=dump)
    ref = ct.load_ctscene(dump)
    fs = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    assert ref.geometry_digest() == fs.geometry_digest() and ref.bvh_digest() == fs.bvh_digest()


@pytest.mark.parametrize("threads", ["1", "3", "8"])
def test_threaded_ingest_and_build_match_the_sequential_reference_algorithms(threads, tmp_path, monkeypatch):
    """PLY import and BVH build on several host threads (SURVEY 8f row f1) give, value for value and node for node,
    what one thread gives -- which the tests above tie to the reference's parser and BuildBVH.  A mesh big enough
    to take the threaded paths (> 50k PLY lines, > 16k triangles), checked against the oracle's BuildBVH restatement."""
    parts = procedural.small_standin_parts(6)             # 8 * 4^6 = 32768 triangles in the largest part
    scene, n = procedural.write_dragon_standin(str(tmp_path), parts=parts, name="mid")
    assert n > 40000
    monkeypatch.setenv("CT_HOST_THREADS", threads)
    fs = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    monkeypatch.setenv("CT_HOST_THREADS", "1")
    one = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    assert fs.geometry_digest() == one.geometry_digest() and fs.bvh_digest() == one.bvh_digest()
    if threads == "8":
        b = O.build_bvh(fs.tri)
        assert all(np.array_equal(v, getattr(fs, k)) for k, v in b.items())
    # the order-exact scatter form of the reference's partition (split_node_parallel, tools/partition_closed_form.py),
    # forced onto every node above the task grain
    monkeypatch.setenv("CT_HOST_THREADS", "4" if threads == "1" else threads)
    monkeypatch.setenv("CT_HOST_PAR_PARTITION_MIN", "3")
    par = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    assert par.bvh_digest() == one.bvh_digest()


@pytest.mark.parametrize("style", ["crlf", "blank_lines", "indented", "no_final_newline", "short_line"])
def test_threaded_ply_import_on_untidy_files(style, tmp_path, monkeypatch, capfd):
    """The threaded PLY import finds its records by the rule of the reference's walk (take the leading numbers of a line,
    skip to the first non-space character after the line end) in slices of the file: CRLF line ends, blank lines,
    indented and padded lines and a missing final newline must give what the one-thread walk gives; a vertex line that
    is too short makes the record run into the next line -- then the sequential walk takes over, same (odd) result."""
    rng = np.random.default_rng(7)
    nv, nf = 30000, 30000                               # 60000 records: above the threaded path's threshold
    verts = rng.normal(size=(nv, 3)).round(4)
    faces = rng.integers(0, nv, size=(nf, 3))
    eol = "\r\n" if style == "crlf" else "\n"
    lines = ["ply", "format ascii 1.0", f"element vertex {nv}", "property float x", "property float y", "property float z",
             f"element face {nf}", "property list uchar int vertex_indices", "end_header"]
    for i, v in enumerate(verts):
        text = f"{v[0]} {v[1]} {v[2]}"
        if style == "indented":
            text = " " * (i % 3) + text + " " * (i % 4) + ("\t" if i % 5 == 0 else "")
        if style == "short_line" and i == 12345:
            text = f"{v[0]} {v[1]}"
        lines.append(text)
        if style == "blank_lines" and i % 7 == 0:
            lines.extend(["", "   "][: 1 + i % 2])
    for f in faces:
        lines.append(f"3 {f[0]} {f[1]} {f[2]}")
    body = eol.join(lines) + ("" if style == "no_final_newline" else eol)
    os.makedirs(tmp_path / "models")
    (tmp_path / "models" / "m.ply").write_text(body, newline="")
    (tmp_path / "s.json").write_text('{"settings": {"numberOfThreads": 2}, "camera": {"position": [0, 0, -8]}, "lights": [{"type": "ambient", "intensity": 0.5}],'
                                     ' "objects": [{"type": "import", "format": "ply", "filename": "models/m.ply", "position": [0, 0, 0], "rotation": [0, 0, 0],'
                                     ' "scale": [1, 1, 1], "color": [255, 255, 255], "specular": 10, "reflection": 0}]}')
    digests = []
    monkeypatch.setenv("CT_HOST_TIMING", "1")
    for threads in ("1", "5", "8"):
        monkeypatch.setenv("CT_HOST_THREADS", threads)
        try:
            fs = host.HostScene.load(str(tmp_path / "s.json"), base_dir=str(tmp_path)).to_flat(with_bvh=False)
            digests.append((fs.n_tri, fs.geometry_digest()))
        except RuntimeError as e:
            digests.append(("error", str(e)))
    assert digests[0] == digests[1] == digests[2], digests
    log = [ln for ln in capfd.readouterr().err.splitlines() if ln.startswith("import_ply:")]
    assert len(log) == 3 and "declined" in log[0]                  # one thread: always the sequential walk
    if style != "short_line":
        assert digests[0][0] == nf
        assert all(", threaded:" in ln for ln in log[1:]), log       # the threaded path really ran
    else:
        assert all("declined" in ln for ln in log[1:]), log


def test_boss_fails_loudly_without_gpu(scene_loader):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    hs = host.HostScene.from_flat(scene_loader("scene_file_cube"))
    with pytest.raises(RuntimeError) as e:
        host.Boss(hs, 64, 64)
    assert "no CPU fallback" in str(e.value) or "no CUDA device" in str(e.value)


# ---- controls (SURVEY 8f row f4): the event queue + HandleKeyboard + HandleUpdates' camera state ----------------

def _replay(ctl, session):
    """Feed a golden session the way oracle/ref_driver.cpp --session does; yields the camera after every tick."""
    assert ctl.update()                              # tick 0: the first frame, before any key is read
    yield ctl.camera()
    for batch in session.split("|"):
        ctl.keys(batch + "m")                        # the harness appends 'm' so the reference always re-dispatches
        assert ctl.update() and ctl.pending == 0
        yield ctl.camera()


def test_controls_follow_reference_keyboard_sessions(golden, scene_loader):
    assert len(golden["sessions"]) >= 4
    for case, m in golden["sessions"].items():
        ctl = host.Controls(host.HostScene.from_flat(scene_loader(m["scene"])))
        cams = list(_replay(ctl, m["session"]))
        assert len(cams) == len(m["ticks"]) and ctl.frames == len(cams)
        for k, ((pos, _, rot), t) in enumerate(zip(cams, m["ticks"])):
            assert np.array_equal(pos, np.array(t["pos"])), (case, k)      # doubles stepped by 0.1: bit-exact
            assert np.array_equal(rot, np.array(t["rot"])), (case, k)      # float yaw/pitch/roll, float cos/sin


def test_controls_queue_and_redraw_rules(scene_loader):
    hs = host.HostScene.from_flat(scene_loader("scene_file_cube"))
    ctl = host.Controls(hs, event_capacity=4)
    pos0 = ctl.camera()[0].copy()
    ctl.keys("wd")                                   # queued before the first frame ...
    assert ctl.update() and ctl.pending == 2         # ... and not read by it (raythread.cpp:548,557: `changesMade || ...`)
    assert np.array_equal(ctl.camera()[0], pos0)
    assert ctl.update() and ctl.pending == 0         # second tick reads them
    assert np.array_equal(ctl.camera()[0], pos0 + np.array([0.1, 0.1, 0.0]))
    assert not ctl.update() and ctl.frames == 2      # nothing pending -> no new frame
    ctl.keys("xz ")                                  # unbound keys are consumed without a redraw
    assert not ctl.update() and ctl.pending == 0
    ctl.key("w", host.EVENT_KEY_UP)                  # only ET_KEY_DOWN counts (:392)
    assert not ctl.update()
    ctl.key("m")                                     # logs, changes nothing, still a redraw (:424-429)
    assert ctl.update() and np.array_equal(ctl.camera()[0], pos0 + np.array([0.1, 0.1, 0.0]))
    ctl.keys("yyyy")
    with pytest.raises(RuntimeError, match="queue full"):
        ctl.key("y")
    assert ctl.update()
    yaw = np.float32(0)
    for _ in range(4):
        yaw = np.float32(np.float64(yaw) + math.pi / 4 / 4)          # float += double, :417
    assert ctl.camera()[1][0] == yaw
    ctl.keys("c")
    assert ctl.update()
    pos, ypr, rot = ctl.camera()
    assert not pos.any() and not ypr.any() and np.array_equal(rot, np.array([1, 0, 0, 0, 1, 0, 0, 0, 1.0]))
    for _ in range(3):                               # the ring wraps
        ctl.keys("adad"); assert ctl.update()
    assert ctl.pending == 0


def test_random_scene_files_parse_and_build_like_the_reference(golden, tmp_path):
    """The 20 generated scene files of make_golden_fuzz.py through the host parser, BVH builder and controls: triangles,
    materials, lights, BVH and the camera after the recorded key presses equal what the compiled reference produced
    from the same text (GetNumber's fp32 digit accumulation on several number notations, colour truncation, ...)."""
    from conftest import load_fuzz_case
    for k, m in golden["fuzz"].items():
        ref, g = load_fuzz_case(k)
        p = tmp_path / f"s{k}.json"
        p.write_text(g["json"])
        hs = host.HostScene.load(str(p))
        fs = hs.to_flat(with_bvh=True)
        assert fs.n_tri == m["n_tri"] and fs.n_lights == m["n_lights"]
        import dataclasses
        moved = dataclasses.replace(fs, cam_pos=ref.cam_pos, cam_rot=ref.cam_rot)      # the dump holds the camera AFTER the key presses
        assert moved.geometry_digest() == ref.geometry_digest(), k
        assert fs.bvh_digest() == ref.bvh_digest(), k
        ctl = host.Controls(hs)
        assert ctl.update()
        ctl.keys(g["keys"] + "m")
        assert ctl.update()
        pos, _, rot = ctl.camera()
        assert np.array_equal(pos, ref.cam_pos) and np.array_equal(rot, ref.cam_rot), k


def test_write_ppm_channel_order(tmp_path):
    """0x00BBGGRR (PutPixel, draw2d.h:8-20) -> P6 bytes R, G, B."""
    bm = np.array([[0x00112233, 0x000000FF], [0x0000FF00, 0x00FF0000], [0, 0xFFFFFFFF]], np.uint32)
    p = str(tmp_path / "f.ppm")
    host.write_ppm(p, bm)
    data = open(p, "rb").read()
    assert data.startswith(b"P6\n2 3\n255\n")
    px = np.frombuffer(data[len(b"P6\n2 3\n255\n"):], np.uint8).reshape(3, 2, 3)
    assert px[0, 0].tolist() == [0x33, 0x22, 0x11] and px[0, 1].tolist() == [255, 0, 0]
    assert px[1, 0].tolist() == [0, 255, 0] and px[1, 1].tolist() == [0, 0, 255] and px[2, 1].tolist() == [255, 255, 255]
    with pytest.raises(RuntimeError):
        host.write_ppm(str(tmp_path / "no" / "such" / "dir.ppm"), bm)


def test_boss_refuses_subsampling_on_several_devices(golden):
    """settings.subsampling writes into the row below a partition (raythread.cpp:512-531): the boss keeps such a frame on
    one device instead of racing on the seam between devices (and says so before touching any GPU)."""
    from cobbletrace_b200 import api, host
    from conftest import load_golden_scene
    hs = host.HostScene.from_flat(load_golden_scene("scene_file_cube", golden).without_bvh())
    with pytest.raises(RuntimeError, match="whole frame on one device"):
        host.Boss(hs, 64, 64, devices=(0, 1), flags=api.CT_FLAG_SUBSAMPLING)
    with pytest.raises(RuntimeError, match="whole frame on one device"):
        host.Boss(hs, 64, 64, devices=(0,), flags=api.CT_FLAG_SUBSAMPLING, shared_counter="ct_test_subsample", rank=0, world_size=2)


def test_scene_shared_through_posix_shm_is_the_same_scene(golden):
    """ct_host_scene_share / _attach (one parse + one BVH build per box in a multi-GPU job): the attached copy has the
    shared scene's triangles, materials, lights, camera and BVH, bit for bit."""
    from cobbletrace_b200 import host
    from conftest import load_golden_scene
    fs = load_golden_scene("scene_import_bunny", golden).with_reflection(0.25)
    a = host.HostScene.from_flat(fs)
    name = f"ct_test_scene_{os.getpid()}"
    a.share(name)
    try:
        b = host.HostScene.attach(name)
    finally:
        host.HostScene.unshare(name)
    fa, fb = a.to_flat(with_bvh=True), b.to_flat(with_bvh=True)
    assert fa.geometry_digest() == fb.geometry_digest() and fa.bvh_digest() == fb.bvh_digest() == golden["scenes"]["scene_import_bunny"]["bvh_sha256"]
    assert np.array_equal(fa.mat_reflection, fb.mat_reflection) and np.array_equal(fa.cam_rot, fb.cam_rot) and np.array_equal(fa.light_pos, fb.light_pos)
    with pytest.raises(RuntimeError, match="shm_open"):
        host.HostScene.attach(name)                          # unshared: gone
