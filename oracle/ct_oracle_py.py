"""ctypes binding of oracle/_build/libct_oracle.so -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this.
The product package (cobbletrace_b200) must never import it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libct_oracle.so")
REF_DIR = os.path.join(HERE, "_ref")
# The reference's own sources (a checkout of jeng/CobbleTrace), which this repository does not carry: oracle/Makefile
# compiles them into REF_DIR when CT_REFERENCE_SRC names them.
REF_SRC = os.environ.get("CT_REFERENCE_SRC", "")


class _Scene(C.Structure):
    _fields_ = [("n_tri", C.c_uint32), ("n_lights", C.c_uint32), ("n_nodes", C.c_uint32), ("_pad", C.c_uint32),
                ("tri", C.c_void_p), ("mat_color", C.c_void_p), ("mat_specular", C.c_void_p), ("mat_reflection", C.c_void_p),
                ("light_type", C.c_void_p), ("light_intensity", C.c_void_p), ("light_pos", C.c_void_p), ("light_dir", C.c_void_p),
                ("cam_pos", C.c_double * 3), ("cam_rot", C.c_double * 9),
                ("node_min", C.c_void_p), ("node_max", C.c_void_p),
                ("node_left", C.c_void_p), ("node_first", C.c_void_p), ("node_count", C.c_void_p), ("tri_index", C.c_void_p)]


class Counters(C.Structure):
    _fields_ = [("rays_primary", C.c_uint64), ("rays_shadow", C.c_uint64), ("rays_reflection", C.c_uint64),
                ("box_tests", C.c_uint64), ("tri_tests", C.c_uint64),
                ("box_tests_kind", C.c_uint64 * 3), ("tri_tests_kind", C.c_uint64 * 3),
                ("ray_hist", (C.c_uint64 * 32) * 3), ("box_hist", (C.c_uint64 * 32) * 3)]

    def as_dict(self, by_kind=False):
        d = {k: int(getattr(self, k)) for k, _ in self._fields_[:5]}
        if by_kind:
            for i, kind in enumerate(("primary", "shadow", "reflection")):
                d[f"box_tests_{kind}"] = int(self.box_tests_kind[i]); d[f"tri_tests_{kind}"] = int(self.tri_tests_kind[i])
                d[f"ray_hist_{kind}"] = [int(x) for x in self.ray_hist[i]]; d[f"box_hist_{kind}"] = [int(x) for x in self.box_hist[i]]
        return d


WIDE, SUBSAMPLE, SUPERSAMPLE = 1, 2, 4     # ct_oracle_render flags (ct_oracle.h)
HIT_DT = np.dtype([("found", "<u4"), ("index", "<u4"), ("t", "<f4")])

_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(os.path.join(HERE, "ct_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.ct_oracle_build_bvh.restype = C.c_uint32
        L.ct_oracle_build_bvh.argtypes = [C.c_uint32] + [C.c_void_p] * 7
        L.ct_oracle_render.restype = C.c_int
        L.ct_oracle_render.argtypes = [C.POINTER(_Scene), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.POINTER(Counters), C.c_int]
        L.ct_oracle_camera_rotation.argtypes = [C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.ct_oracle_intersect_triangle.restype = C.c_int
        L.ct_oracle_intersect_triangle.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_void_p]
        L.ct_oracle_intersect_aabb.restype = C.c_int
        L.ct_oracle_intersect_aabb.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
        L.ct_oracle_prehit_check.restype = C.c_uint64
        L.ct_oracle_prehit_check.argtypes = [C.POINTER(_Scene), C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        L.ct_oracle_free_check.restype = C.c_uint64
        L.ct_oracle_free_check.argtypes = [C.POINTER(_Scene), C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.ct_oracle_closest.restype = C.c_int
        L.ct_oracle_closest.argtypes = [C.POINTER(_Scene), C.c_void_p, C.c_void_p, C.c_float, C.POINTER(C.c_uint32), C.POINTER(C.c_float)]
        L.ct_oracle_shade_color.restype = C.c_uint32
        L.ct_oracle_shade_color.argtypes = [C.c_uint32, C.c_float]
        L.ct_oracle_blend.restype = C.c_uint32
        L.ct_oracle_blend.argtypes = [C.c_uint32, C.c_uint32, C.c_float]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def build_bvh(tri: np.ndarray):
    """Restated BuildBVH (bvh.cpp:16-120). Returns dict of node arrays + tri_index."""
    tri = np.ascontiguousarray(tri, np.float64).reshape(-1, 9)
    n = tri.shape[0]
    cap = max(2 * n - 1, 1)
    nmin = np.zeros((cap, 3)); nmax = np.zeros((cap, 3))
    left = np.zeros(cap, np.uint32); first = np.zeros(cap, np.uint32); count = np.zeros(cap, np.uint32)
    index = np.zeros(max(n, 1), np.uint32)
    used = lib().ct_oracle_build_bvh(n, _ptr(tri), _ptr(nmin), _ptr(nmax), _ptr(left), _ptr(first), _ptr(count), _ptr(index))
    return dict(node_min=nmin[:used].copy(), node_max=nmax[:used].copy(), node_left=left[:used].copy(),
                node_first=first[:used].copy(), node_count=count[:used].copy(), tri_index=index[:n].copy())


class OracleScene:
    """Keeps the numpy arrays alive behind a ct_oracle_scene struct."""

    def __init__(self, fs):
        if not fs.has_bvh():
            import dataclasses
            fs = dataclasses.replace(fs, **build_bvh(fs.tri))
        self.fs = fs
        keep = {}
        def c(name, dtype):
            keep[name] = np.ascontiguousarray(getattr(fs, name), dtype)
            return _ptr(keep[name])
        s = _Scene()
        s.n_tri, s.n_lights, s.n_nodes = fs.n_tri, fs.n_lights, fs.n_nodes
        s.tri = c("tri", np.float64)
        s.mat_color = c("mat_color", np.uint32); s.mat_specular = c("mat_specular", np.int32); s.mat_reflection = c("mat_reflection", np.float32)
        s.light_type = c("light_type", np.int32); s.light_intensity = c("light_intensity", np.float32)
        s.light_pos = c("light_pos", np.float64); s.light_dir = c("light_dir", np.float64)
        s.cam_pos = (C.c_double * 3)(*np.asarray(fs.cam_pos, np.float64).tolist())
        s.cam_rot = (C.c_double * 9)(*np.asarray(fs.cam_rot, np.float64).tolist())
        s.node_min = c("node_min", np.float64); s.node_max = c("node_max", np.float64)
        s.node_left = c("node_left", np.uint32); s.node_first = c("node_first", np.uint32); s.node_count = c("node_count", np.uint32)
        s.tri_index = c("tri_index", np.uint32)
        self._keep = keep
        self.c = s

    def render(self, W, H, y_start=None, y_end=None, max_depth=10, flags=0, want_hits=True, n_threads=None, by_kind=False):
        half = H // 2      # HandleUpdates raythread.cpp:574-581 with a thread count dividing H: rows [-(H/2), -(H/2)+H)
        y_start = -half if y_start is None else y_start
        y_end = -half + H if y_end is None else y_end
        frame = np.zeros((H, W), np.uint32)
        hits = None
        if want_hits:
            hits = np.zeros((H, W), HIT_DT)
            hits["found"] = 0xFFFFFFFF
        ctr = Counters()
        n_threads = n_threads or min(os.cpu_count() or 1, 32)
        lib().ct_oracle_render(C.byref(self.c), W, H, y_start, y_end, max_depth, flags, _ptr(frame),
                               _ptr(hits) if hits is not None else None, C.byref(ctr), n_threads)
        return frame, hits, ctr.as_dict(by_kind)

    def closest(self, org, direction, t0=1e30):
        org = np.ascontiguousarray(org, np.float64); direction = np.ascontiguousarray(direction, np.float64)
        idx = C.c_uint32(); t = C.c_float()
        found = lib().ct_oracle_closest(C.byref(self.c), _ptr(org), _ptr(direction), np.float32(t0), C.byref(idx), C.byref(t))
        return bool(found), int(idx.value), float(t.value)

    def closest_many(self, org, direction, t0=1e30):
        """closest() for n rays in one call: (found, index, t) arrays."""
        org = np.ascontiguousarray(org, np.float64).reshape(-1, 3); direction = np.ascontiguousarray(direction, np.float64).reshape(-1, 3)
        n = org.shape[0]
        t0 = np.ascontiguousarray(np.broadcast_to(np.asarray(t0, np.float32), (n,)))
        found = np.zeros(n, np.uint32); index = np.zeros(n, np.uint32); t = np.zeros(n, np.float32)
        L = lib()
        L.ct_oracle_closest_many.restype = None
        L.ct_oracle_closest_many.argtypes = [C.POINTER(_Scene), C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ct_oracle_closest_many(C.byref(self.c), n, _ptr(org), _ptr(direction), _ptr(t0), _ptr(found), _ptr(index), _ptr(t))
        return found, index, t


def prehit_check(scene: "OracleScene", org, direction):
    """Prototype check (ct_oracle.c): reference-order closest-hit walk vs "order-free pre-hit phase + rebuilt stack"
    over the given rays.  Returns (rays that differ, rays that found something)."""
    org = np.ascontiguousarray(org, np.float64); direction = np.ascontiguousarray(direction, np.float64)
    found = C.c_uint64()
    bad = lib().ct_oracle_prehit_check(C.byref(scene.c), org.shape[0], _ptr(org), _ptr(direction), C.byref(found))
    return int(bad), int(found.value)


def free_check(scene: "OracleScene", org, direction, order=1):
    """Prototype check (ct_oracle.c): reference-order closest-hit walk vs the order-free walk + candidate replay.
    Returns (rays that differ, stats dict)."""
    org = np.ascontiguousarray(org, np.float64); direction = np.ascontiguousarray(direction, np.float64)
    st = np.zeros(4, np.uint64); ref = np.zeros(2, np.uint64)
    bad = lib().ct_oracle_free_check(C.byref(scene.c), org.shape[0], _ptr(org), _ptr(direction), order, _ptr(st), _ptr(ref))
    return int(bad), {"box": int(st[0]), "tri": int(st[1]), "fallback": int(st[2]), "max_cand": int(st[3]),
                      "ref_box": int(ref[0]), "ref_tri": int(ref[1]), "rays": int(org.shape[0])}


def rounds_check(scene: "OracleScene", org, direction, min_visits=0):
    """Prototype (ct_oracle.c): the order-free closest-hit search as a 32-wide frontier against the reference-order walk, for the rays
    whose ordered walk needs >= min_visits pair visits."""
    org = np.ascontiguousarray(org, np.float64); direction = np.ascontiguousarray(direction, np.float64)
    out = np.zeros(8, np.uint64)
    L = lib()
    L.ct_oracle_rounds_check.restype = None
    L.ct_oracle_rounds_check.argtypes = [C.POINTER(_Scene), C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.ct_oracle_rounds_check(C.byref(scene.c), org.shape[0], _ptr(org), _ptr(direction), min_visits, _ptr(out))
    keys = ("rays", "differ", "undecided", "ordered_pair_visits", "rounds", "max_ordered_pair_visits", "max_rounds", "rounds_of_longest")
    return {k: int(v) for k, v in zip(keys, out)}


def slop_check(org, direction, tri):
    """(passes, max (tmin(box of the triangle) - t) / M, skipped) over (ray, triangle) cases, all in the reference's arithmetic."""
    org = np.ascontiguousarray(org, np.float64); direction = np.ascontiguousarray(direction, np.float64)
    tri = np.ascontiguousarray(tri, np.float64).reshape(-1, 9)
    out = np.zeros(3)
    L = lib()
    L.ct_oracle_slop_check.restype = None
    L.ct_oracle_slop_check.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.ct_oracle_slop_check(org.shape[0], _ptr(org), _ptr(direction), _ptr(tri), _ptr(out))
    return int(out[0]), float(out[1]), int(out[2])


def camera_rotation(yaw=0.0, pitch=0.0, roll=0.0):
    out = np.zeros(9)
    lib().ct_oracle_camera_rotation(yaw, pitch, roll, _ptr(out))
    return out


# ---- oracle/_ref (the compiled, unmodified reference) ---------------------------------------------

def ref_available() -> bool:
    return os.path.exists(os.path.join(REF_DIR, "ct_ref"))


def run_ref(scene_json, chdir=None, width=640, height=640, depth=10, threads=8, force_reflection=None,
            frame=None, hits=None, dump_scene=None, time_frames=0, counters=False, timeout=3600):
    """Run oracle/_ref/ct_ref[_count]; returns its JSON line as dict."""
    import json
    exe = os.path.join(REF_DIR, "ct_ref_count" if counters else "ct_ref")
    cmd = [exe, "--scene", scene_json, "--width", str(width), "--height", str(height), "--depth", str(depth),
           "--threads", str(threads)]
    if chdir: cmd += ["--chdir", chdir]
    if force_reflection is not None: cmd += ["--force-reflection", repr(float(force_reflection))]
    if frame: cmd += ["--frame", frame]
    if hits: cmd += ["--hits", hits]
    if dump_scene: cmd += ["--dump-scene", dump_scene]
    if time_frames: cmd += ["--time", str(time_frames)]
    if counters: cmd += ["--counters"]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=timeout).stdout
    return json.loads(out.strip().splitlines()[-1])
