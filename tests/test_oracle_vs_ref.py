"""Live cross-check: the plain-C restatement against the compiled, unmodified reference (oracle/_ref).
Skipped where the reference's sources (CT_REFERENCE_SRC) were not available at build time; the committed goldens cover that case."""
import os

import numpy as np
import pytest

import cobbletrace_b200 as ct
from oracle import ct_oracle_py as O

pytestmark = pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref not built (needs the reference's sources: CT_REFERENCE_SRC)")
SCENES = os.path.join(O.REF_DIR, "scenes")


@pytest.mark.parametrize("scene,W,H,depth,refl,threads", [
    ("scene_file_cube.json", 320, 320, 10, None, 8),
    ("scene_file_cube.json", 300, 200, 4, 0.7, 4),
    ("scene_import.json", 200, 200, 10, None, 8),
    ("scene_import_bunny.json", 256, 256, 10, None, 8),
    ("scene_import_bunny.json", 192, 192, 3, 0.4, 6),
    ("pc_big.json", 64, 64, 10, None, 4),
])
def test_restatement_equals_reference(tmp_path, scene, W, H, depth, refl, threads):
    fr, hi, du = (str(tmp_path / n) for n in ("f.bin", "h.bin", "s.ctscene"))
    info = O.run_ref(scene, chdir=SCENES, width=W, height=H, depth=depth, threads=threads, force_reflection=refl,
                     frame=fr, hits=hi, dump_scene=du, counters=True)
    fs = ct.load_ctscene(du)
    if refl is not None:
        fs = fs.with_reflection(refl)
    ref_frame = np.fromfile(fr, np.uint32).reshape(H, W)
    ref_hits = np.fromfile(hi, O.HIT_DT).reshape(H, W)
    frame, hits, ctr = O.OracleScene(fs).render(W, H, max_depth=depth)
    assert np.array_equal(frame, ref_frame)
    assert np.array_equal(hits["found"], ref_hits["found"])
    tr = ref_hits["found"] != 0xFFFFFFFF
    assert np.array_equal(hits["index"][tr], ref_hits["index"][tr])
    assert np.array_equal(hits["t"][tr].view(np.uint32), ref_hits["t"][tr].view(np.uint32))
    for k in ("rays_primary", "rays_shadow", "rays_reflection", "box_tests", "tri_tests"):
        assert ctr[k] == info[k], k


def test_reference_drops_rows_when_threads_do_not_divide_height(tmp_path):
    """raythread.cpp:576: yStep = H / numberOfThreads in integers -- 100 rows over 8 threads leaves 4 rows unrendered."""
    fr = str(tmp_path / "f.bin")
    O.run_ref("scene_file_cube.json", chdir=SCENES, width=100, height=100, threads=8, frame=fr)
    frame = np.fromfile(fr, np.uint32).reshape(100, 100)
    assert int((frame == 0).all(axis=1).sum()) == 1 + 4        # row 0 plus the 4 lost rows
