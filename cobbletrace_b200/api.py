"""ctypes binding of the C ABI in include/ct_gpu.h (libct_gpu.so).

This is the reference-facing plugin call path: host buffers in, host framebuffer out.  There is no
CPU fallback -- if the CUDA library is missing or no device is present every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from .sceneio import FlatScene

PKG = os.path.dirname(os.path.abspath(__file__))
GPU_LIB = os.path.join(PKG, "libct_gpu.so")

CT_FLAG_WIDE, CT_FLAG_KEEP_HITS, CT_FLAG_COUNT_TESTS, CT_FLAG_STAGE_TIMING, CT_FLAG_SUBSAMPLING, CT_FLAG_SUPERSAMPLING = 1, 2, 4, 8, 16, 32
CT_FLAG_BUILD_BVH = 64
BACKGROUND = 0x333333      # raythread.cpp:59
REFERENCE_MAX_DEPTH = 10   # raythread.cpp:508

# every symbol include/ct_gpu.h declares
ABI_SYMBOLS = [
    "ct_gpu_abi_version", "ct_gpu_device_count", "ct_gpu_last_error", "ct_gpu_upload_scene", "ct_gpu_set_camera",
    "ct_gpu_set_stream", "ct_gpu_render_tile", "ct_gpu_readback", "ct_gpu_readback_async", "ct_gpu_readback_wait", "ct_gpu_readback_hits", "ct_gpu_get_counters",
    "ct_gpu_last_tile_ms", "ct_gpu_sync", "ct_gpu_throttle", "ct_gpu_kernel_launches", "ct_gpu_last_tile_stages", "ct_gpu_framebuffer", "ct_gpu_gather_rows", "ct_gpu_debug_closest", "ct_gpu_debug_early", "ct_gpu_debug_primary",
    "ct_gpu_debug_primitives", "ct_gpu_debug_filter", "ct_gpu_filter_stats", "ct_gpu_reuse_stats", "ct_gpu_shutdown", "ct_gpu_share_export", "ct_gpu_share_attach", "ct_gpu_share_reset", "ct_gpu_share_partition", "ct_gpu_mark_rows", "ct_gpu_render_shared", "ct_gpu_set_option", "ct_gpu_overflow_stats",
    "ct_gpu_build_bvh", "ct_gpu_debug_scene_array", "ct_gpu_trace_rays", "ct_gpu_shade_rays", "ct_gpu_update_triangles", "ct_gpu_debug_shading",
    "ct_gpu_update_scene",
]
CT_UPDATE_TRIANGLES, CT_UPDATE_MATERIALS, CT_UPDATE_LIGHTS = 1, 2, 4
RAY_KINDS = {"primary": 0, "shadow": 1, "reflection": 2}     # CT_RAY_PRIMARY, CT_RAY_SHADOW, CT_RAY_REFLECTION


class CtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ct_gpu error {code}: {msg}")
        self.code = code


class BvhNode(C.Structure):      # == ct_bvh_node == reference bvh_node_t (bvh.h:5-11)
    _fields_ = [("aabb_min", C.c_double * 3), ("aabb_max", C.c_double * 3), ("left_node", C.c_uint32),
                ("first_triangle_index", C.c_uint32), ("triangle_count", C.c_uint32), ("_pad", C.c_uint32)]


class Material(C.Structure):     # == ct_material == reference material_t (scenefile.h:25-29)
    _fields_ = [("color", C.c_uint32), ("specular", C.c_int32), ("reflection", C.c_float)]


class Light(C.Structure):        # == ct_light == reference light_t (scenefile.h:61-66)
    _fields_ = [("type", C.c_int32), ("intensity", C.c_float), ("position", C.c_double * 3), ("direction", C.c_double * 3)]


class Share(C.Structure):        # == ct_gpu_share
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("pid", C.c_int64), ("fb_ptr", C.c_uint64), ("cursor_ptr", C.c_uint64),
                ("fb_ipc", C.c_ubyte * 64), ("cursor_ipc", C.c_ubyte * 64), ("width", C.c_int32), ("height", C.c_int32), ("frames", C.c_uint64)]


class SceneDesc(C.Structure):    # == ct_scene_desc
    _fields_ = [("struct_size", C.c_uint32), ("flags", C.c_uint32),
                ("n_triangles", C.c_uint32), ("triangle_stride", C.c_uint32),
                ("triangles", C.c_void_p), ("materials", C.c_void_p),
                ("n_nodes", C.c_uint32), ("n_lights", C.c_uint32),
                ("nodes", C.c_void_p), ("tri_indexes", C.c_void_p), ("lights", C.c_void_p),
                ("camera_position", C.c_double * 3), ("camera_rotation", C.c_double * 9), ("viewport", C.c_float * 3),
                ("width", C.c_int32), ("height", C.c_int32), ("max_depth", C.c_int32), ("background", C.c_uint32)]


class RayQuery(C.Structure):     # == ct_ray_query
    _fields_ = [("struct_size", C.c_uint32), ("kind", C.c_int32), ("n", C.c_uint32), ("_pad", C.c_uint32),
                ("origins", C.c_void_p), ("directions", C.c_void_p), ("found", C.c_void_p), ("index", C.c_void_p),
                ("tclosest", C.c_void_p), ("stream", C.c_void_p)]


class ShadeQuery(C.Structure):   # == ct_shade_query
    _fields_ = [("struct_size", C.c_uint32), ("n", C.c_uint32), ("max_depth", C.c_int32), ("_pad", C.c_uint32),
                ("origins", C.c_void_p), ("directions", C.c_void_p), ("color", C.c_void_p), ("stream", C.c_void_p)]


class TriangleUpdate(C.Structure):   # == ct_triangle_update
    _fields_ = [("struct_size", C.c_uint32), ("n_triangles", C.c_uint32), ("triangle_stride", C.c_uint32), ("_pad", C.c_uint32),
                ("triangles", C.c_void_p), ("stream", C.c_void_p)]


class SceneUpdate(C.Structure):  # == ct_scene_update
    _fields_ = [("struct_size", C.c_uint32), ("what", C.c_uint32), ("n_triangles", C.c_uint32), ("triangle_stride", C.c_uint32),
                ("n_lights", C.c_uint32), ("_pad", C.c_uint32), ("triangles", C.c_void_p), ("materials", C.c_void_p),
                ("lights", C.c_void_p), ("stream", C.c_void_p)]


class PathSummary(C.Structure):  # == ct_path_summary (ct_gpu_debug_scene_array "path_state")
    _fields_ = [(k, C.c_uint32) for k in ("n_triangles", "n_lights", "n_shadow_lights", "occ_words", "any_leaves", "any_reflective",
                                          "levels", "ovf_cap")]


class RayCounters(C.Structure):  # == ct_ray_counters
    _fields_ = [("rays_primary", C.c_uint64), ("rays_shadow", C.c_uint64), ("rays_reflection", C.c_uint64),
                ("box_tests", C.c_uint64), ("tri_tests", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


NODE_DT = np.dtype([("min", "<f8", 3), ("max", "<f8", 3), ("left", "<u4"), ("first", "<u4"), ("count", "<u4"), ("pad", "<u4")])
MAT_DT = np.dtype([("color", "<u4"), ("specular", "<i4"), ("reflection", "<f4")])
LIGHT_DT = np.dtype([("type", "<i4"), ("intensity", "<f4"), ("pos", "<f8", 3), ("dir", "<f8", 3)])
assert NODE_DT.itemsize == C.sizeof(BvhNode) == 64 and MAT_DT.itemsize == C.sizeof(Material) == 12
assert LIGHT_DT.itemsize == C.sizeof(Light) == 56
# == ct_scene_summary (ct_gpu_debug_scene_array "summary")
SUMMARY_DT = np.dtype([("n_pairs", "<u4"), ("n_wide", "<u4"), ("root_ref", "<u4"), ("root_cnt", "<u4"), ("pos_of_tri0", "<u4"), ("nested", "<u4"),
                       ("leaf_dfs_order", "<u4"), ("can_overflow", "<u4"), ("bound", "<f8", 3), ("depth", "<i4"), ("pad", "<u4")])
assert SUMMARY_DT.itemsize == 64
SCENE_ARRAYS = ("wide", "pairs32", "pairs64", "tris32", "tris", "materials", "pair_parent", "tri_parent", "summary")
# == ct_path_summary (ct_gpu_debug_scene_array "path_state")
PATH_DT = np.dtype([(k, "<u4") for k, _ in PathSummary._fields_])
assert PATH_DT.itemsize == C.sizeof(PathSummary) == 32
# everything a loaded scene's frames read: the arrays, the device's light records and what the path state was sized from
SCENE_STATE = SCENE_ARRAYS + ("lights", "shadow_lights", "path_state")

_lib = None


def load_library(path: Optional[str] = None):
    """Load libct_gpu.so (no fallback: a missing library is an error)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or GPU_LIB
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found: build it with `python -m cobbletrace_b200.build` "
                           "(cobbletrace_b200 is CUDA-only; there is no CPU fallback)")
    L = C.CDLL(path)
    vp = C.c_void_p
    L.ct_gpu_last_error.restype = C.c_char_p
    L.ct_gpu_upload_scene.argtypes = [C.c_int, C.POINTER(SceneDesc)]
    L.ct_gpu_set_camera.argtypes = [C.c_int, vp, vp]
    L.ct_gpu_set_stream.argtypes = [C.c_int, vp]
    L.ct_gpu_render_tile.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(RayCounters)]
    L.ct_gpu_readback.argtypes = [C.c_int, vp, C.c_int, C.c_int, C.c_int]
    L.ct_gpu_readback_async.argtypes = [C.c_int, vp, C.c_int, C.c_int, C.c_int]
    L.ct_gpu_readback_wait.argtypes = [C.c_int]
    L.ct_gpu_readback_hits.argtypes = [C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int]
    L.ct_gpu_get_counters.argtypes = [C.c_int, C.POINTER(RayCounters), C.c_int]
    L.ct_gpu_last_tile_ms.argtypes = [C.c_int, C.POINTER(C.c_float)]
    L.ct_gpu_sync.argtypes = [C.c_int]
    L.ct_gpu_throttle.argtypes = [C.c_int, C.c_int]
    L.ct_gpu_kernel_launches.argtypes = [C.c_int, C.POINTER(C.c_uint64), C.c_int]
    L.ct_gpu_last_tile_stages.argtypes = [C.c_int, C.c_int, vp, vp, vp]
    L.ct_gpu_framebuffer.argtypes = [C.c_int, C.POINTER(vp), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.ct_gpu_gather_rows.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    L.ct_gpu_debug_closest.argtypes = [C.c_int, C.c_uint32, vp, vp, vp, vp, vp, vp]
    L.ct_gpu_debug_early.argtypes = [C.c_int, C.c_int, C.c_uint32, vp, vp, vp, vp, vp]
    L.ct_gpu_debug_primary.argtypes = [C.c_int, C.c_uint32, vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.ct_gpu_debug_primitives.argtypes = [C.c_int, C.c_uint32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.ct_gpu_debug_filter.argtypes = [C.c_int, C.c_uint32, vp, vp, vp, vp, vp, vp, C.c_double, vp]
    L.ct_gpu_debug_shading.argtypes = [C.c_int, C.c_uint32] + [vp] * 13
    L.ct_gpu_filter_stats.argtypes = [C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.ct_gpu_reuse_stats.argtypes = [C.c_int, C.POINTER(C.c_uint64)]
    L.ct_gpu_share_export.argtypes = [C.c_int, C.POINTER(Share)]
    L.ct_gpu_share_attach.argtypes = [C.c_int, C.POINTER(Share)]
    L.ct_gpu_share_reset.argtypes = [C.c_int]
    L.ct_gpu_share_partition.argtypes = [C.c_int, C.c_int, C.c_int]
    L.ct_gpu_mark_rows.argtypes = [C.c_int, C.c_int, C.c_int]
    L.ct_gpu_render_shared.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(RayCounters)]
    L.ct_gpu_shutdown.argtypes = [C.c_int]
    L.ct_gpu_set_option.argtypes = [C.c_char_p, C.c_longlong]
    L.ct_gpu_overflow_stats.argtypes = [C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.ct_gpu_build_bvh.argtypes = [C.c_int, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp]
    L.ct_gpu_debug_scene_array.argtypes = [C.c_int, C.c_char_p, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.ct_gpu_trace_rays.argtypes = [C.c_int, C.POINTER(RayQuery)]
    L.ct_gpu_shade_rays.argtypes = [C.c_int, C.POINTER(ShadeQuery)]
    L.ct_gpu_update_triangles.argtypes = [C.c_int, C.POINTER(TriangleUpdate)]
    L.ct_gpu_update_scene.argtypes = [C.c_int, C.POINTER(SceneUpdate)]
    if path == GPU_LIB:
        _lib = L
    return L


def _check(L, rc: int):
    if rc < 0:
        raise CtError(rc, L.ct_gpu_last_error().decode(errors="replace"))
    return rc


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pack_nodes(fs: FlatScene) -> np.ndarray:
    n = np.zeros(fs.n_nodes, NODE_DT)
    n["min"], n["max"] = fs.node_min, fs.node_max
    n["left"], n["first"], n["count"] = fs.node_left, fs.node_first, fs.node_count
    return n


class GpuRenderer:
    """One device's renderer: upload once, render row tiles, read back (SURVEY 8b)."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        self.device = int(device)
        self.width = self.height = 0
        self.flags = 0
        self.n_tri = None

    # -- ct_gpu_upload_scene ------------------------------------------------------------------------
    def upload(self, fs: FlatScene, width: int, height: int, max_depth: int = REFERENCE_MAX_DEPTH, flags: int = 0,
               background: int = BACKGROUND, viewport=(1.0, 1.0, 1.0), triangle_stride: int = 72, build_bvh: bool = False):
        """`triangle_stride` = 96 lays the vertices out like the reference's triangle_t (scenefile.h:36-41: p1, p2, p3 and
        a centroid the tracer never reads -- filled with NaNs here so that a wrong stride cannot go unnoticed).
        `build_bvh`: the device builds the reference's tree from the triangles (CT_FLAG_BUILD_BVH); a tree `fs` carries is ignored."""
        if build_bvh:
            flags |= CT_FLAG_BUILD_BVH
        elif not fs.has_bvh():
            raise ValueError("FlatScene has no BVH: build it on the host first (cobbletrace_b200.host.build_bvh)")
        tri = np.ascontiguousarray(fs.tri, np.float64)
        if triangle_stride != 72:
            wide = np.full((fs.n_tri, triangle_stride // 8), np.nan)
            wide[:, :9] = tri.reshape(fs.n_tri, 9)
            tri = wide
        mats = np.zeros(fs.n_tri, MAT_DT)
        mats["color"], mats["specular"], mats["reflection"] = fs.mat_color, fs.mat_specular, fs.mat_reflection
        lights = np.zeros(max(fs.n_lights, 1), LIGHT_DT)
        if fs.n_lights:
            lights["type"][:fs.n_lights], lights["intensity"][:fs.n_lights] = fs.light_type, fs.light_intensity
            lights["pos"][:fs.n_lights], lights["dir"][:fs.n_lights] = fs.light_pos, fs.light_dir
        nodes = None if build_bvh else pack_nodes(fs)
        idx = None if build_bvh else np.ascontiguousarray(fs.tri_index, np.uint32)
        d = SceneDesc()
        d.struct_size = C.sizeof(SceneDesc)
        d.flags = flags
        d.n_triangles, d.triangle_stride = fs.n_tri, triangle_stride
        d.triangles, d.materials = _ptr(tri), _ptr(mats)
        d.n_nodes, d.n_lights = (0 if build_bvh else fs.n_nodes), fs.n_lights
        d.nodes, d.tri_indexes, d.lights = _ptr(nodes), _ptr(idx), _ptr(lights)
        d.camera_position = (C.c_double * 3)(*np.asarray(fs.cam_pos, np.float64).tolist())
        d.camera_rotation = (C.c_double * 9)(*np.asarray(fs.cam_rot, np.float64).tolist())
        d.viewport = (C.c_float * 3)(*viewport)
        d.width, d.height, d.max_depth, d.background = width, height, max_depth, background
        _check(self.L, self.L.ct_gpu_upload_scene(self.device, C.byref(d)))
        self.width, self.height, self.flags, self.n_tri = width, height, flags, fs.n_tri
        return self

    # -- ct_gpu_update_triangles ----------------------------------------------------------------------
    def update_triangles(self, triangles):
        """Replace the loaded scene's triangles and rebuild the reference's tree over them on the device, in place: afterwards the
        device holds the scene upload(..., build_bvh=True) would load from them with the scene's materials, lights, camera and frame;
        the stream set with set_stream, the framebuffer, counters and shared-frame state stay.  See ct_gpu_update_triangles.

        torch tensor: float64, shape (n, 9) or (n, 3, 3) (p1, p2, p3 per triangle), contiguous, on cuda:<device>, n the uploaded
        scene's triangle count.  It is read in place in torch.cuda.current_stream(device)'s order, so a kernel that wrote it on that
        stream needs no synchronisation; the call returns when the update is done.  numpy array: copied to the device first.
        Anything else raises ValueError before the library is called."""
        import torch
        dev = torch.device("cuda", self.device)
        triangles = self._device_triangles(triangles, dev)
        if self.n_tri is not None and triangles.shape[0] != self.n_tri:
            raise ValueError(f"{triangles.shape[0]} triangles: the uploaded scene has {self.n_tri}")
        u = TriangleUpdate()
        u.struct_size, u.n_triangles, u.triangle_stride = C.sizeof(TriangleUpdate), triangles.shape[0], 72
        u.triangles = triangles.data_ptr() or None
        u.stream = torch.cuda.current_stream(dev).cuda_stream or 1      # (handle 0, torch's default stream, is cudaStreamLegacy = 1)
        _check(self.L, self.L.ct_gpu_update_triangles(self.device, C.byref(u)))

    @staticmethod
    def _device_triangles(triangles, dev):
        """The triangles update_triangles / update_scene read in place: a float64 (n, 9) or (n, 3, 3) contiguous tensor on `dev`
        (numpy: copied there)."""
        import torch
        if isinstance(triangles, np.ndarray):
            triangles = torch.from_numpy(np.ascontiguousarray(triangles, np.float64)).to(dev)
        if not isinstance(triangles, torch.Tensor):
            raise ValueError(f"triangles: a torch tensor or a numpy array, not {type(triangles).__name__}")
        if triangles.device != dev:
            raise ValueError(f"triangles are on {triangles.device}, this renderer's scene is on {dev}")
        if triangles.dtype != torch.float64:
            raise ValueError(f"triangles are {triangles.dtype}, vertices are float64")
        if tuple(triangles.shape[1:]) not in ((9,), (3, 3)):
            raise ValueError(f"triangles have shape {tuple(triangles.shape)}, not (n, 9) or (n, 3, 3)")
        if not triangles.is_contiguous():
            raise ValueError("triangles are not contiguous")
        return triangles

    @staticmethod
    def _columns(what, parts, names, dtypes, widths, dev):
        """A tuple of tensors on `dev`, one per record field: 1-D (width 0) or (n, width), of the given dtypes, of one length n."""
        import torch
        if not isinstance(parts, (tuple, list)) or len(parts) != len(names):
            raise ValueError(f"{what}: a numpy record array or a tuple ({', '.join(names)}) of tensors")
        n = None
        for name, a, ok, w in zip(names, parts, dtypes, widths):
            if not isinstance(a, torch.Tensor):
                raise ValueError(f"{what} {name}: a torch tensor, not {type(a).__name__}")
            if a.device != dev:
                raise ValueError(f"{what} {name} is on {a.device}, this renderer's scene is on {dev}")
            if a.dtype not in ok:
                raise ValueError(f"{what} {name} is {a.dtype}, not {' or '.join(map(str, ok))}")
            if a.shape[1:] != ((w,) if w else ()) or a.dim() != (2 if w else 1):
                raise ValueError(f"{what} {name} has shape {tuple(a.shape)}, not (n{', %d' % w if w else ''})")
            if n is not None and a.shape[0] != n:
                raise ValueError(f"{what}: {name} has {a.shape[0]} entries, {names[0]} {n}")
            n = a.shape[0]
        return n

    def _device_materials(self, materials, dev):
        """ct_material records (12 bytes) on `dev`: from a numpy MAT_DT array (copied), or packed on the current stream from
        (color uint32 or int64 -- its low 32 bits --, specular int32, reflection float32) tensors."""
        import torch
        if isinstance(materials, np.ndarray):
            if materials.dtype != MAT_DT or materials.ndim != 1:
                raise ValueError(f"materials: a 1-D array of api.MAT_DT, not {materials.dtype} of shape {materials.shape}")
            return torch.from_numpy(np.ascontiguousarray(materials).view(np.uint8)).to(dev).view(-1, 12), materials.shape[0]
        n = self._columns("materials", materials, ("color", "specular", "reflection"),
                          ((torch.uint32, torch.int64), (torch.int32,), (torch.float32,)), (0, 0, 0), dev)
        color, specular, reflection = materials
        if color.dtype == torch.int64:
            color = color & 0xFFFFFFFF
            color = torch.where(color >= 2**31, color - 2**32, color).to(torch.int32)
        else:
            color = color.view(torch.int32)
        return torch.stack([color, specular, reflection.view(torch.int32)], 1).contiguous(), n

    def _device_lights(self, lights, dev):
        """ct_light records (56 bytes) on `dev`: from a numpy LIGHT_DT array (copied), or packed on the current stream from
        (type int32 or int64, intensity float32, pos float64 (n, 3), dir float64 (n, 3)) tensors."""
        import torch
        if isinstance(lights, np.ndarray):
            if lights.dtype != LIGHT_DT or lights.ndim != 1:
                raise ValueError(f"lights: a 1-D array of api.LIGHT_DT, not {lights.dtype} of shape {lights.shape}")
            return torch.from_numpy(np.ascontiguousarray(lights).view(np.uint8)).to(dev).view(-1, 56), lights.shape[0]
        n = self._columns("lights", lights, ("type", "intensity", "pos", "dir"),
                          ((torch.int32, torch.int64), (torch.float32,), (torch.float64,), (torch.float64,)), (0, 0, 3, 3), dev)
        ltype, intensity, pos, direction = lights
        if n == 0:
            return torch.empty((0, 56), dtype=torch.uint8, device=dev), 0
        parts = [(ltype.to(torch.int32), 4), (intensity, 4), (pos, 24), (direction, 24)]      # ct_light: type, intensity, position, direction
        return torch.cat([a.contiguous().view(torch.uint8).view(n, w) for a, w in parts], 1), n

    # -- ct_gpu_update_scene --------------------------------------------------------------------------
    def update_scene(self, triangles=None, materials=None, lights=None):
        """Replace any of the loaded scene's triangles (of any count), materials and lights from device memory: afterwards the device
        holds the scene upload(..., build_bvh=True) would load from the new parts and the loaded ones left out, with the scene's camera
        and frame; the stream set with set_stream, the framebuffer, counters and shared-frame state stay.  See ct_gpu_update_scene.

        triangles: as update_triangles takes them, of any count; a new count needs new materials too.
        materials: a numpy MAT_DT array, or a (color, specular, reflection) tuple of 1-D tensors on cuda:<device> -- color uint32 or
                   int64 (its low 32 bits, 0x00BBGGRR), specular int32, reflection float32 -- one per triangle, by triangle id.
        lights:    a numpy LIGHT_DT array, or a (type, intensity, pos, dir) tuple of tensors on cuda:<device> -- type int32 or int64,
                   intensity float32, pos and dir float64 (n, 3) -- in file order; an empty one removes every light.
        Tensors are packed into the library's records on torch.cuda.current_stream(device) and read in that stream's order, so a
        kernel that wrote them there needs no synchronisation; numpy arrays are copied to the device first.  The call returns when the
        update is done.  Anything malformed raises ValueError before the library is called."""
        import torch
        if triangles is None and materials is None and lights is None:
            raise ValueError("update_scene: give triangles, materials or lights")
        dev = torch.device("cuda", self.device)
        u = SceneUpdate()
        u.struct_size = C.sizeof(SceneUpdate)
        keep = []                                                       # the packed inputs live until the call returns
        n = self.n_tri
        if triangles is not None:
            t = self._device_triangles(triangles, dev)
            u.what |= CT_UPDATE_TRIANGLES
            n, u.triangle_stride, u.triangles = t.shape[0], 72, t.data_ptr() or None
            if n == 0:
                raise ValueError("triangles: a scene has at least one triangle")
            keep.append(t)
        if materials is not None:
            m, n_mat = self._device_materials(materials, dev)
            if n_mat != n:
                raise ValueError(f"{n_mat} materials for {n} triangles")
            u.what |= CT_UPDATE_MATERIALS
            u.materials = m.data_ptr() or None
            keep.append(m)
        elif n != self.n_tri:
            raise ValueError(f"{n} triangles: the uploaded scene has {self.n_tri}; a new count needs new materials")
        u.n_triangles = n or 0
        if lights is not None:
            lt, n_lit = self._device_lights(lights, dev)
            u.what |= CT_UPDATE_LIGHTS
            u.n_lights, u.lights = n_lit, (lt.data_ptr() or None) if n_lit else None
            keep.append(lt)
        u.stream = torch.cuda.current_stream(dev).cuda_stream or 1      # (handle 0, torch's default stream, is cudaStreamLegacy = 1)
        _check(self.L, self.L.ct_gpu_update_scene(self.device, C.byref(u)))
        self.n_tri = n

    def set_camera(self, position, rotation):
        p = np.ascontiguousarray(position, np.float64); r = np.ascontiguousarray(rotation, np.float64).reshape(9)
        _check(self.L, self.L.ct_gpu_set_camera(self.device, _ptr(p), _ptr(r)))

    def set_stream(self, cuda_stream_ptr: Optional[int]):
        _check(self.L, self.L.ct_gpu_set_stream(self.device, C.c_void_p(cuda_stream_ptr or 0)))

    # -- ct_gpu_render_tile ---------------------------------------------------------------------------
    def full_range(self):
        half = self.height // 2
        # HandleUpdates raythread.cpp:574-581 with a thread count that divides H: yStart = -(H/2),
        # yEnd = yStart + N * (H/N) = yStart + H  (H/2 for even H; odd H also reaches row 0)
        return -half, -half + self.height

    def render_tile(self, y_start: Optional[int] = None, y_end: Optional[int] = None, counters: bool = False):
        if y_start is None:
            y_start, y_end = self.full_range()
        c = RayCounters() if counters else None
        _check(self.L, self.L.ct_gpu_render_tile(self.device, y_start, y_end, C.byref(c) if counters else None))
        return c.as_dict() if counters else None

    # -- one frame on several GPUs (ct_gpu_share_*) ------------------------------------------------------------
    def share_export(self) -> bytes:
        """Root GPU: the handle (plain bytes) the other GPUs attach to."""
        h = Share()
        h.struct_size = C.sizeof(Share)
        _check(self.L, self.L.ct_gpu_share_export(self.device, C.byref(h)))
        return bytes(h)

    def share_attach(self, handle: Optional[bytes]):
        if handle is None:
            _check(self.L, self.L.ct_gpu_share_attach(self.device, None))
            return
        h = Share.from_buffer_copy(handle)
        _check(self.L, self.L.ct_gpu_share_attach(self.device, C.byref(h)))

    def mark_rows(self, row_start: int, row_end: int):
        """Framebuffer rows filled from outside the library (e.g. multi.gather_rows_to_root): readback must cover them."""
        _check(self.L, self.L.ct_gpu_mark_rows(self.device, row_start, row_end))

    def share_partition(self, index: int, count: int):
        """This GPU is participant `index` of `count` in every shared frame (ct_gpu_share_partition)."""
        _check(self.L, self.L.ct_gpu_share_partition(self.device, index, count))

    def share_reset(self):
        _check(self.L, self.L.ct_gpu_share_reset(self.device))

    def render_shared(self, y_start: Optional[int] = None, y_end: Optional[int] = None, counters: bool = False):
        if y_start is None:
            y_start, y_end = self.full_range()
        c = RayCounters() if counters else None
        _check(self.L, self.L.ct_gpu_render_shared(self.device, y_start, y_end, C.byref(c) if counters else None))
        return c.as_dict() if counters else None

    def sync(self):
        _check(self.L, self.L.ct_gpu_sync(self.device))

    def last_tile_ms(self) -> float:
        ms = C.c_float()
        _check(self.L, self.L.ct_gpu_last_tile_ms(self.device, C.byref(ms)))
        return float(ms.value)

    def kernel_launches(self, reset: bool = False) -> int:
        n = C.c_uint64()
        _check(self.L, self.L.ct_gpu_kernel_launches(self.device, C.byref(n), int(reset)))
        return int(n.value)

    def last_tile_stages(self):
        """[(kernel name, depth, ms)] of the last tile (needs CT_FLAG_STAGE_TIMING)."""
        ms = (C.c_float * 80)(); names = (C.c_char_p * 80)(); depth = (C.c_int * 80)()
        n = _check(self.L, self.L.ct_gpu_last_tile_stages(self.device, 80, ms, names, depth))
        return [(names[i].decode(), int(depth[i]), float(ms[i])) for i in range(n)]

    def counters(self, reset: bool = False):
        c = RayCounters()
        _check(self.L, self.L.ct_gpu_get_counters(self.device, C.byref(c), int(reset)))
        return c.as_dict()

    # -- ct_gpu_readback ------------------------------------------------------------------------------
    def readback(self, out: Optional[np.ndarray] = None, row_start: int = 0, row_end: Optional[int] = None) -> np.ndarray:
        if out is None:
            out = np.zeros((self.height, self.width), np.uint32)   # calloc'd like cobbletrace.cpp:57
        assert out.dtype == np.uint32 and out.flags.c_contiguous and out.shape[0] >= self.height
        row_end = self.height if row_end is None else row_end
        _check(self.L, self.L.ct_gpu_readback(self.device, _ptr(out), out.shape[1], row_start, row_end))
        return out

    def readback_async(self, out: np.ndarray, row_start: int = 0, row_end: Optional[int] = None) -> None:
        """ct_gpu_readback_async: `out` (page-locked for a truly asynchronous copy) is filled by readback_wait()."""
        assert out.dtype == np.uint32 and out.flags.c_contiguous and out.shape[0] >= self.height
        row_end = self.height if row_end is None else row_end
        _check(self.L, self.L.ct_gpu_readback_async(self.device, _ptr(out), out.shape[1], row_start, row_end))

    def readback_wait(self) -> None:
        _check(self.L, self.L.ct_gpu_readback_wait(self.device))

    def readback_hits(self):
        H, W = self.height, self.width
        found = np.zeros((H, W), np.uint32); index = np.zeros((H, W), np.uint32); t = np.zeros((H, W), np.float32)
        _check(self.L, self.L.ct_gpu_readback_hits(self.device, _ptr(found), _ptr(index), _ptr(t), W, 0, H))
        return found, index, t

    def framebuffer_ptr(self):
        p = C.c_void_p(); w = C.c_int(); h = C.c_int()
        _check(self.L, self.L.ct_gpu_framebuffer(self.device, C.byref(p), C.byref(w), C.byref(h)))
        return int(p.value), int(w.value), int(h.value)

    def gather_rows_to(self, dst_device: int, row_start: int, row_end: int):
        _check(self.L, self.L.ct_gpu_gather_rows(self.device, dst_device, row_start, row_end))

    def _check_rays(self, origins, directions, dev):
        """The rays trace_rays / shade_rays read in place: float64 (n, 3) contiguous tensors on this renderer's device."""
        import torch
        for name, a in (("origins", origins), ("directions", directions)):
            if not isinstance(a, torch.Tensor):
                raise ValueError(f"{name}: a torch tensor or a numpy array, not {type(a).__name__}")
            if a.device != dev:
                raise ValueError(f"{name} is on {a.device}, this renderer traces on {dev}")
            if a.dtype != torch.float64:
                raise ValueError(f"{name} is {a.dtype}, rays are float64")
            if a.dim() != 2 or a.shape[1] != 3:
                raise ValueError(f"{name} has shape {tuple(a.shape)}, rays are (n, 3)")
            if not a.is_contiguous():
                raise ValueError(f"{name} is not contiguous")
        if origins.shape != directions.shape:
            raise ValueError(f"origins {tuple(origins.shape)} and directions {tuple(directions.shape)} differ in shape")

    # -- ct_gpu_trace_rays ----------------------------------------------------------------------------
    def trace_rays(self, origins, directions, kind: str = "primary"):
        """ClosestIntersection for n rays of one kind the reference casts ("primary": ray.t = 1e30f, the closest hit; "shadow":
        occlusion; "reflection": ray.t = 0, the first barycentric pass in DFS order), bit for bit; see ct_gpu_trace_rays.
        Returns (found, index, tclosest), None for what the kind does not define (shadow rays: found only).

        torch tensors: float64, shape (n, 3), contiguous, on cuda:<device>.  They are read in place, the work runs on
        torch.cuda.current_stream(device), and the results are int32 / float32 tensors on the device that are valid in that
        stream's order: the call does not synchronise.  numpy arrays: copied to the device, traced, synchronised, returned as
        numpy (found / index uint32, tclosest float32)."""
        import torch
        if kind not in RAY_KINDS:
            raise ValueError(f"kind must be one of {sorted(RAY_KINDS)}, not {kind!r}")
        dev = torch.device("cuda", self.device)
        if isinstance(origins, np.ndarray) and isinstance(directions, np.ndarray):
            o = torch.from_numpy(np.ascontiguousarray(origins, np.float64).reshape(-1, 3)).to(dev)
            d = torch.from_numpy(np.ascontiguousarray(directions, np.float64).reshape(-1, 3)).to(dev)
            out = self.trace_rays(o, d, kind)
            torch.cuda.current_stream(dev).synchronize()
            found, index, t = (None if x is None else x.cpu().numpy() for x in out)
            return (found.view(np.uint32), None if index is None else index.view(np.uint32), t)
        self._check_rays(origins, directions, dev)
        n = origins.shape[0]
        found = torch.empty(n, dtype=torch.int32, device=dev)
        index = None if kind == "shadow" else torch.empty(n, dtype=torch.int32, device=dev)
        t = None if kind == "shadow" else torch.empty(n, dtype=torch.float32, device=dev)
        q = RayQuery()
        q.struct_size, q.kind, q.n = C.sizeof(RayQuery), RAY_KINDS[kind], n
        q.origins, q.directions = origins.data_ptr() or None, directions.data_ptr() or None
        q.found = found.data_ptr() or None
        q.index = None if index is None else (index.data_ptr() or None)
        q.tclosest = None if t is None else (t.data_ptr() or None)
        q.stream = torch.cuda.current_stream(dev).cuda_stream or 1      # (handle 0, torch's default stream, is cudaStreamLegacy = 1)
        _check(self.L, self.L.ct_gpu_trace_rays(self.device, C.byref(q)))
        return found, index, t

    # -- ct_gpu_shade_rays ----------------------------------------------------------------------------
    def shade_rays(self, origins, directions, max_depth: Optional[int] = None):
        """TraceRay's colour (0x00BBGGRR) for n rays: lighting, shadow rays and `max_depth` levels of reflection (None: the depth
        the scene was uploaded with), bit for bit; a miss gets the background.  See ct_gpu_shade_rays.

        torch tensors: float64, shape (n, 3), contiguous, on cuda:<device>.  They are read in place, the work runs on
        torch.cuda.current_stream(device), and the colours come back as an int32 tensor on the device that is valid in that stream's
        order: the call does not synchronise.  numpy arrays: copied to the device, shaded, synchronised, returned as uint32 numpy.
        Anything else raises ValueError, as trace_rays does."""
        import torch
        if max_depth is not None and (not isinstance(max_depth, (int, np.integer)) or isinstance(max_depth, bool) or not -2**31 <= max_depth < 2**31):
            raise ValueError(f"max_depth must be an int or None, not {max_depth!r}")
        dev = torch.device("cuda", self.device)
        if isinstance(origins, np.ndarray) and isinstance(directions, np.ndarray):
            o = torch.from_numpy(np.ascontiguousarray(origins, np.float64).reshape(-1, 3)).to(dev)
            d = torch.from_numpy(np.ascontiguousarray(directions, np.float64).reshape(-1, 3)).to(dev)
            color = self.shade_rays(o, d, max_depth)
            torch.cuda.current_stream(dev).synchronize()
            return color.cpu().numpy().view(np.uint32)
        self._check_rays(origins, directions, dev)
        n = origins.shape[0]
        color = torch.empty(n, dtype=torch.int32, device=dev)
        q = ShadeQuery()
        q.struct_size, q.n, q.max_depth = C.sizeof(ShadeQuery), n, -1 if max_depth is None else int(max_depth)
        q.origins, q.directions, q.color = origins.data_ptr() or None, directions.data_ptr() or None, color.data_ptr() or None
        q.stream = torch.cuda.current_stream(dev).cuda_stream or 1      # (handle 0, torch's default stream, is cudaStreamLegacy = 1)
        _check(self.L, self.L.ct_gpu_shade_rays(self.device, C.byref(q)))
        return color

    # -- KAT entry points -----------------------------------------------------------------------------
    def debug_closest(self, origins, directions, t0):
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3); d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        n = o.shape[0]
        t0 = np.ascontiguousarray(np.broadcast_to(np.asarray(t0, np.float32), (n,)))
        found = np.zeros(n, np.uint32); index = np.zeros(n, np.uint32); t = np.zeros(n, np.float32)
        _check(self.L, self.L.ct_gpu_debug_closest(self.device, n, _ptr(o), _ptr(d), _ptr(t0), _ptr(found), _ptr(index), _ptr(t)))
        return found, index, t

    def debug_early(self, origins, directions, mode):
        """ct_gpu_debug_early: mode 0 = shadow rays (found = occluded), 1 = reflection rays (index = first pass in DFS order).
        Returns (found, index, path) with path 0 own walk, 1 k_overflow, 2 k_overflow_huge, 3 finished in place."""
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3); d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        n = o.shape[0]
        found = np.zeros(n, np.uint32); index = np.zeros(n, np.uint32); path = np.zeros(n, np.uint32)
        _check(self.L, self.L.ct_gpu_debug_early(self.device, int(mode), n, _ptr(o), _ptr(d), _ptr(found), _ptr(index), _ptr(path)))
        return found, index, path

    def debug_primary(self, origins, directions, park_cap=0):
        """ct_gpu_debug_primary: primary rays (ray.t = 1e30f) along a frame's path.  Returns (found, index, tclosest, path); path & 0xff:
        0 own walk, 1 k_primary_long, 2 k_primary_split, 3 in place; path >> 8: k_primary_split's outcome (0 = decided by its frontier)."""
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3); d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        n = o.shape[0]
        found = np.zeros(n, np.uint32); index = np.zeros(n, np.uint32); t = np.zeros(n, np.float32); path = np.zeros(n, np.uint32)
        _check(self.L, self.L.ct_gpu_debug_primary(self.device, n, _ptr(o), _ptr(d), int(park_cap), _ptr(found), _ptr(index), _ptr(t), _ptr(path)))
        return found, index, t, path

    def debug_primitives(self, origins, directions, ray_t, tri, bmin, bmax):
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3); d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        n = o.shape[0]
        rt = np.ascontiguousarray(np.broadcast_to(np.asarray(ray_t, np.float32), (n,))).copy()
        tri = np.ascontiguousarray(tri, np.float64).reshape(n, 9)
        mn = np.ascontiguousarray(bmin, np.float64).reshape(n, 3); mx = np.ascontiguousarray(bmax, np.float64).reshape(n, 3)
        th = np.zeros(n, np.uint32); bh = np.zeros(n, np.uint32)
        _check(self.L, self.L.ct_gpu_debug_primitives(self.device, n, _ptr(o), _ptr(d), _ptr(rt), _ptr(tri), _ptr(mn), _ptr(mx), _ptr(th), _ptr(bh)))
        return th, bh, rt

    def debug_filter(self, origins, directions, ray_t, bmin, bmax, bound_scale=1.0, tri=None):
        """ct_gpu_debug_filter: verdict codes of the certified fp32 filters next to the reference's verdicts."""
        o = np.ascontiguousarray(origins, np.float64); d = np.ascontiguousarray(directions, np.float64)
        rt = np.ascontiguousarray(ray_t, np.float32)
        mn = np.ascontiguousarray(bmin, np.float64); mx = np.ascontiguousarray(bmax, np.float64)
        tr = None if tri is None else np.ascontiguousarray(tri, np.float64)
        n = o.shape[0]
        out = np.zeros(n, np.uint32)
        _check(self.L, self.L.ct_gpu_debug_filter(self.device, n, _ptr(o), _ptr(d), _ptr(rt), _ptr(tr), _ptr(mn), _ptr(mx), float(bound_scale), _ptr(out)))
        return out

    def debug_shading(self, color=None, intensity=None, lc=None, rc=None, reflection=None, x=None, e=None, acc=None, li=None):
        """ct_gpu_debug_shading: the shading arithmetic on independent cases.  Each family is computed when its inputs are given:
        (color, intensity) -> shaded uint32, (lc, rc, reflection) -> blended uint32, (x, e) -> pow float64, and with (acc, li) too the
        specular accumulation float32.  Returns a dict of the families computed."""
        u32 = lambda a: None if a is None else np.ascontiguousarray(a, np.uint32).ravel()
        f32 = lambda a: None if a is None else np.ascontiguousarray(a, np.float32).ravel()
        ins = dict(color=u32(color), intensity=f32(intensity), lc=u32(lc), rc=u32(rc), reflection=f32(reflection), x=f32(x),
                   e=None if e is None else np.ascontiguousarray(e, np.int32).ravel(), acc=f32(acc), li=f32(li))
        sizes = {a.size for a in ins.values() if a is not None}
        if len(sizes) != 1:
            raise ValueError("debug_shading: give at least one family, every input of the same length")
        n = sizes.pop()
        fam = {"shaded": ("color", "intensity"), "blended": ("lc", "rc", "reflection"), "pow": ("x", "e"), "acc": ("x", "e", "acc", "li")}
        out = {k: np.zeros(n, np.float64 if k == "pow" else np.float32 if k == "acc" else np.uint32)
               for k, need in fam.items() if all(ins[a] is not None for a in need)}
        _check(self.L, self.L.ct_gpu_debug_shading(self.device, n, _ptr(ins["color"]), _ptr(ins["intensity"]), _ptr(out.get("shaded")),
                                                   _ptr(ins["lc"]), _ptr(ins["rc"]), _ptr(ins["reflection"]), _ptr(out.get("blended")),
                                                   _ptr(ins["x"]), _ptr(ins["e"]), _ptr(out.get("pow")), _ptr(ins["acc"]), _ptr(ins["li"]),
                                                   _ptr(out.get("acc"))))
        return out

    def debug_scene_array(self, name: str) -> np.ndarray:
        """ct_gpu_debug_scene_array: the bytes of one array the upload built (api.SCENE_STATE); "summary" as a SUMMARY_DT record,
        "path_state" as a PATH_DT record."""
        n = C.c_size_t()
        _check(self.L, self.L.ct_gpu_debug_scene_array(self.device, name.encode(), None, 0, C.byref(n)))
        out = np.zeros(n.value, np.uint8)
        _check(self.L, self.L.ct_gpu_debug_scene_array(self.device, name.encode(), _ptr(out), out.size, C.byref(n)))
        if name == "summary":
            return out.view(SUMMARY_DT)[0]
        return out.view(PATH_DT)[0] if name == "path_state" else out

    def filter_stats(self):
        """(box tests, triangle tests) the fp32 filters left to the fp64 arithmetic (needs CT_FLAG_COUNT_TESTS)."""
        a = C.c_uint64(); b = C.c_uint64()
        _check(self.L, self.L.ct_gpu_filter_stats(self.device, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def reuse_stats(self) -> int:
        """Shadow rays (counted in rays_shadow) answered from an ancestor's identical ray instead of being traced."""
        a = C.c_uint64()
        _check(self.L, self.L.ct_gpu_reuse_stats(self.device, C.byref(a)))
        return int(a.value)

    def overflow_stats(self):
        """(rays parked for the breadth-first overflow kernel, rays finished in place because the buffer was full)."""
        a = C.c_uint64(); b = C.c_uint64()
        _check(self.L, self.L.ct_gpu_overflow_stats(self.device, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def shutdown(self):
        _check(self.L, self.L.ct_gpu_shutdown(self.device))


def set_option(name: str, value: int) -> None:
    """ct_gpu_set_option: library-wide knob applied by the next upload (e.g. "traversal_budget")."""
    L = load_library()
    _check(L, L.ct_gpu_set_option(name.encode(), int(value)))


def build_bvh(fs: FlatScene, device: int = 0, triangle_stride: int = 72) -> FlatScene:
    """`fs` with the node arrays and tri_index of the reference's BuildBVH, built on `device` by ct_gpu_build_bvh.
    `triangle_stride` lays the triangles out as GpuRenderer.upload does."""
    import dataclasses
    L = load_library()
    n = fs.n_tri
    tri = np.ascontiguousarray(fs.tri, np.float64).reshape(n, 9)
    if triangle_stride != 72:
        wide = np.full((n, triangle_stride // 8), np.nan)
        wide[:, :9] = tri
        tri = wide
    nodes = np.zeros(max(2 * n - 1, 1), NODE_DT)
    idx = np.zeros(max(n, 1), np.uint32)
    used = _check(L, L.ct_gpu_build_bvh(int(device), n, _ptr(tri), triangle_stride, _ptr(nodes), nodes.shape[0], _ptr(idx)))
    nodes = nodes[:used]
    return dataclasses.replace(fs, node_min=nodes["min"].copy(), node_max=nodes["max"].copy(), node_left=nodes["left"].copy(),
                               node_first=nodes["first"].copy(), node_count=nodes["count"].copy(), tri_index=idx[:n].copy())


def device_count() -> int:
    L = load_library()
    return _check(L, L.ct_gpu_device_count())
