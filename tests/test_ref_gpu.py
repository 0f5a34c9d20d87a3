"""The drop-in, executed: oracle/_ref/ct_ref_gpu is the reference itself (its parser, GetSceneTriangles, BuildBVH,
HandleKeyboard, HandleUpdates -- compiled from the reference's sources named by CT_REFERENCE_SRC) with the two statements
of RayThread that the INTEGRATION.md patch replaces (oracle/ref_gpu_patch.h: worker threads -> ct_gpu_render_tile per
partition, ct_gpu_readback into bitmap->memory), linked against libct_gpu.so.  It hands the reference's arrays over as
they are: bvh_node_t[], light_t[], and triangle_t[] at its real 96-byte stride (scenefile.h:36-41).
The reference's sources are not part of this repository; without them these tests skip.  The library calls the patch
makes (96-byte stride, row tiles, read-back) are checked against the reference's stored frames in test_gpu_parity."""
import os
import subprocess

import numpy as np
import pytest

import cobbletrace_b200 as ct
from oracle import ct_oracle_py as O

EXE = os.path.join(O.REF_DIR, "ct_ref_gpu")
SCENES = os.path.join(O.REF_DIR, "scenes")
FILES = {"scene_file_cube": "scene_file_cube.json", "scene_import": "scene_import.json", "scene_import_bunny": "scene_import_bunny.json",
         "pc_big": "pc_big.json"}


def _built():
    if os.path.isdir(O.REF_SRC):
        from cobbletrace_b200 import build
        build.build_gpu()
        subprocess.check_call(["make", "-s", "-C", os.path.join(os.path.dirname(O.REF_DIR)), "ref", "ref_gpu"])
    if not os.path.exists(EXE):
        pytest.skip("oracle/_ref/ct_ref_gpu not built (needs the reference's sources: CT_REFERENCE_SRC)")


def run_ref_gpu(tmp_path, scene, W, H, depth=10, threads=8, refl=None, keys=None):
    out = str(tmp_path / "gpu_frame.bin")
    cmd = [EXE, "--scene", FILES[scene], "--chdir", SCENES, "--width", str(W), "--height", str(H), "--depth", str(depth),
           "--threads", str(threads), "--frame", out]
    if refl is not None:
        cmd += ["--force-reflection", repr(float(refl))]
    if keys:
        cmd += ["--keys", keys]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    return p, out


def test_reference_binding_compiles_and_has_no_cpu_fallback(tmp_path):
    """`make ref_gpu` compiles the INTEGRATION.md patch against the reference's own sources; without a CUDA device the
    patched reference stops with the library's error instead of rendering anything."""
    _built()
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present: covered by the gpu tests")
    p, out = run_ref_gpu(tmp_path, "scene_file_cube", 64, 64)
    assert p.returncode == 4 and "no CPU fallback" in p.stderr and not os.path.exists(out)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", sorted(FILES))
def test_reference_with_gpu_workers_reproduces_the_reference_frames(scene, golden, tmp_path):
    """640x640, depth 10, 8 partitions (the reference's default thread count): the frame the patched reference leaves in
    bitmap->memory hashes to what the unmodified reference rendered (SURVEY 8c hashes, tests/golden)."""
    _built()
    p, out = run_ref_gpu(tmp_path, scene, 640, 640)
    assert p.returncode == 0, p.stderr
    assert '"triangle_stride": 96' in p.stdout
    frame = np.fromfile(out, np.uint32).reshape(640, 640)
    assert ct.frame_fnv1a(frame) == golden["scenes"][scene]["frame640_fnv1a"], scene
    assert int((frame == 0).sum()) == 640                       # row 0 never written


@pytest.mark.gpu
@pytest.mark.parametrize("scene,W,H,threads,depth,refl,keys", [
    ("scene_file_cube", 200, 120, 7, 10, None, None),       # H % threads != 0: the rows HandleUpdates never hands out stay zero (:576)
    ("scene_import_bunny", 160, 160, 5, 2, 0.5, None),
    ("scene_import", 150, 150, 1, 10, None, "ypw"),         # keys through the reference's own HandleKeyboard / camera matrix
])
def test_patched_reference_equals_unmodified_reference_byte_for_byte(scene, W, H, threads, depth, refl, keys, tmp_path):
    _built()
    assert O.ref_available()
    p, out = run_ref_gpu(tmp_path, scene, W, H, depth=depth, threads=threads, refl=refl, keys=keys)
    assert p.returncode == 0, p.stderr
    want = str(tmp_path / "cpu_frame.bin")
    cmd = [os.path.join(O.REF_DIR, "ct_ref"), "--scene", FILES[scene], "--chdir", SCENES, "--width", str(W), "--height", str(H),
           "--depth", str(depth), "--threads", str(threads), "--frame", want]
    if refl is not None:
        cmd += ["--force-reflection", repr(float(refl))]
    if keys:
        cmd += ["--keys", keys]
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)
    a, b = np.fromfile(out, np.uint32), np.fromfile(want, np.uint32)
    assert a.size == b.size == W * H and np.array_equal(a, b)
