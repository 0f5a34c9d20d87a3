"""ct_gpu_trace_rays / GpuRenderer.trace_rays: primary, shadow and reflection rays held in device memory.

Every answer is checked bit for bit against the oracle's ClosestIntersection (ray.t = 1e30f: primary found / index / tclosest,
shadow found; ray.t = 0: reflection found / index / tclosest) and against the KAT entries ct_gpu_debug_primary / ct_gpu_debug_early,
which run the same path in the caller's order.  Permuting the rays must not change any ray's bits (also with the rays binned
before the walk, build switch -DCT_RAY_BINS=1)."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api, host, procedural
from oracle import ct_oracle_py as O
from test_walk_limits import (FINF, PARK_ALL, axis_rays, comb, gpu, options, ray_families, reverse_leaf_order, soup, spine,  # noqa: F401 (gpu: fixture)
                              stack)

KINDS = ("primary", "shadow", "reflection")
CT_ERR_INVALID, CT_ERR_NO_SCENE, CT_ERR_LIMIT = -1, -4, -5
SETTINGS = {
    "default": {},
    "budget6": dict(traversal_budget=6),                                   # shadow / reflection rays parked for k_overflow
    "warp1": dict(traversal_budget=6, overflow_warp_budget=1),             # ... and handed on to k_overflow_huge
    "long1": dict(primary_budget=1),                                       # primary rays parked for k_primary_long
    "long6": dict(primary_budget=6),
    "split1": dict(primary_budget=1, primary_split=1),                     # ... for k_primary_split
    "split6": dict(primary_budget=6, primary_split=1),
}


def torch_rays(o, d, device=0):
    import torch
    return (torch.from_numpy(np.ascontiguousarray(o, np.float64)).to(f"cuda:{device}"),
            torch.from_numpy(np.ascontiguousarray(d, np.float64)).to(f"cuda:{device}"))


def host_results(res):
    return tuple(None if x is None else x.cpu().numpy() for x in res)


def oracle_answers(fs, o, d):
    osc = O.OracleScene(fs)
    closest, first = osc.closest_many(o, d, 1e30), osc.closest_many(o, d, 0.0)
    return {"primary": closest, "shadow": (closest[0], None, None), "reflection": first}


def assert_same(got, want, what):
    """(found, index, tclosest) against (found, index, tclosest); None in `want` = not defined for the kind (must be None in `got`)."""
    for name, g, w in zip(("found", "index", "tclosest"), got, want):
        if w is None:
            assert g is None, (what, name)
            continue
        g = np.asarray(g).view(np.uint32)
        w = np.asarray(w).astype(np.float32 if name == "tclosest" else np.uint32).view(np.uint32)
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, f"{what} {name}: {bad.size} of {g.size} rays differ, first ray {bad[0]}: {g[bad[0]]:#x} against {w[bad[0]]:#x}"


def trace_all(gpu, ot, dt):
    return {kind: host_results(gpu.trace_rays(ot, dt, kind)) for kind in KINDS}


def debug_answers(gpu, o, d):
    """The KAT entries' answers and path codes: {kind: ((found, index, tclosest), path)}."""
    f, i, t, p = gpu.debug_primary(o, d)
    out = {"primary": ((f, i, t), p)}
    f, i, p = gpu.debug_early(o, d, 0)
    out["shadow"] = ((f, None, None), p)
    f, i, p = gpu.debug_early(o, d, 1)
    out["reflection"] = ((f, i, None), p)
    return out


# ---- 1. oracle parity, every kind, every parking path ------------------------------------------------------------------------
def scene(name, scene_loader, rng):
    if name == "soup":
        return soup(rng)
    if name == "comb96":
        return comb(95, rng)
    if name == "spine":
        return spine(rng)
    if name == "reversed":
        return reverse_leaf_order(soup(rng, 600))
    return scene_loader(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["scene_import_bunny", "pc_big", "scene_file_cube", "scene_import", "soup", "comb96", "spine", "reversed"])
def test_every_kind_matches_the_oracle(name, scene_loader, gpu):
    rng = np.random.default_rng(sum(map(ord, name)) + 4)
    fs = scene(name, scene_loader, rng)
    fam = ray_families(fs, rng, scale=0.4 if name == "scene_import_bunny" else 1.0)
    if name in ("comb96", "spine"):
        fam.update(axis_rays(rng))
    o, d = stack(fam)
    ref = oracle_answers(fs, o, d)
    ot, dt = torch_rays(o, d)
    small = fs.n_nodes + fs.n_tri <= 384                     # a tree this small parks at all only with a small traversal budget
    paths = {kind: set() for kind in KINDS}
    for setting, kw in SETTINGS.items():
        kw = dict(kw, traversal_budget=6) if small and "primary_budget" in kw else kw
        with options(**kw):
            gpu.upload(fs, 32, 32, max_depth=2)
            got = trace_all(gpu, ot, dt)
            for kind in KINDS:
                assert_same(got[kind], ref[kind], f"{name} {setting} {kind}")
            for kind, (res, path) in debug_answers(gpu, o, d).items():
                paths[kind] |= set(np.unique(path & 0xff).tolist())
    # the settings above take the rays through every parking path (the KAT entries' path codes: same rays, same path)
    if name in ("scene_import_bunny", "pc_big", "scene_file_cube", "soup"):
        assert {1, 2} <= paths["shadow"] and {1, 2} <= paths["reflection"] and {1, 2} <= paths["primary"], (name, paths)


# ---- 2. the same path as the KAT entries, at scale -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dragon():
    with tempfile.TemporaryDirectory() as d:
        path, _ = procedural.write_dragon_standin(d)
        bare = host.HostScene.load(path, base_dir=d).to_flat(with_bvh=False)
    return api.build_bvh(bare)


def random_rays(fs, rng, n):
    lo, hi = fs.node_min[0], fs.node_max[0]
    o = lo + (hi - lo) * rng.uniform(-0.3, 1.3, (n, 3))
    d = rng.normal(size=(n, 3))
    return o, d


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["default", "park"])
def test_same_answers_as_the_kat_entries_on_the_dragon_stand_in(setting, dragon, gpu):
    rng = np.random.default_rng(2024)
    o, d = random_rays(dragon, rng, 1 << 20)
    ot, dt = torch_rays(o, d)
    with options(**({} if setting == "default" else PARK_ALL)):
        gpu.upload(dragon, 64, 64, max_depth=2)
        got = trace_all(gpu, ot, dt)
        for kind, (res, _) in debug_answers(gpu, o, d).items():
            want = res if kind != "reflection" else (res[0], res[1], got[kind][2])
            assert_same(got[kind], want, f"dragon {setting} {kind} against the KAT entry")
    sub = rng.choice(len(o), 100_000, replace=False) if setting == "default" else np.arange(0)
    if sub.size:
        ref = oracle_answers(dragon, o[sub], d[sub])
        for kind in KINDS:
            assert_same(tuple(None if x is None else x[sub] for x in got[kind]), ref[kind], f"dragon {kind} against the oracle")


# ---- 3. the order of the rays does not matter ----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_order_does_not_change_any_ray(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny")
    rng = np.random.default_rng(3)
    o, d = random_rays(fs, rng, 200_000)
    ot, dt = torch_rays(o, d)
    for kw in ({}, dict(traversal_budget=6, primary_budget=1, primary_split=1)):
        with options(**kw):
            gpu.upload(fs, 32, 32, max_depth=2)
            base = trace_all(gpu, ot, dt)
            for perm in (torch.randperm(len(o), generator=torch.Generator().manual_seed(5)), torch.arange(len(o) - 1, -1, -1)):
                p = perm.to(ot.device)
                got = trace_all(gpu, ot[p].contiguous(), dt[p].contiguous())
                inv = np.argsort(perm.numpy())
                for kind in KINDS:
                    assert_same(tuple(None if x is None else x[inv] for x in got[kind]), base[kind], f"permuted {kw} {kind}")


# ---- 4. streams and frames ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_results_are_ordered_on_a_torch_side_stream(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_file_cube")
    rng = np.random.default_rng(4)
    o, d = stack(ray_families(fs, rng))
    ref = oracle_answers(fs, o, d)
    gpu.upload(fs, 32, 32)
    ot, dt = torch_rays(o, d)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        f, i, t = gpu.trace_rays(ot, dt, "primary")
        hits = (f * 2 + 1).sum()                      # torch work on the same stream, no host synchronisation in between
        idx = i.clone()
        tt = t.clone()
    side.synchronize()
    assert int(hits) == 2 * int(ref["primary"][0].astype(np.int64).sum()) + len(o)
    assert_same((f.cpu().numpy(), idx.cpu().numpy(), tt.cpu().numpy()), ref["primary"], "side stream")


@pytest.mark.gpu
def test_a_query_between_two_tiles_leaves_the_frame_alone(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_import_bunny").with_reflection(0.5)
    rng = np.random.default_rng(6)
    o, d = stack(ray_families(fs, rng, scale=0.3))
    ref = oracle_answers(fs, o, d)
    ot, dt = torch_rays(o, d)
    W = H = 96
    with options(**PARK_ALL):
        gpu.upload(fs, W, H, max_depth=3, flags=ct.CT_FLAG_COUNT_TESTS)
        gpu.render_tile()
        alone = gpu.readback()
        # queries count nothing: the frame counters, overflow and reuse statistics stay where the frame left them
        before = gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats()
        trace_all(gpu, ot, dt)
        assert (gpu.counters(), gpu.overflow_stats(), gpu.reuse_stats()) == before
        # a query on the render stream between the two tiles of the next frame
        render = torch.cuda.Stream()
        render.wait_stream(torch.cuda.current_stream())
        gpu.set_stream(render.cuda_stream)
        y0, y1 = gpu.full_range()
        with torch.cuda.stream(render):
            gpu.render_tile(y0, (y0 + y1) // 2)
            got = [gpu.trace_rays(ot, dt, kind) for kind in KINDS]
            gpu.render_tile((y0 + y1) // 2, y1)
        gpu.sync()
        gpu.set_stream(None)
        for kind, res in zip(KINDS, got):
            assert_same(host_results(res), ref[kind], f"between tiles {kind}")
        assert np.array_equal(gpu.readback(), alone)


@pytest.mark.gpu
def test_a_query_followed_at_once_by_a_new_upload(scene_loader, gpu):
    fs = scene_loader("pc_big")
    rng = np.random.default_rng(8)
    o, d = random_rays(fs, rng, 100_000)
    ref = oracle_answers(fs, o, d)
    ot, dt = torch_rays(o, d)
    with options(**PARK_ALL):
        gpu.upload(fs, 32, 32)
        got = [gpu.trace_rays(ot, dt, kind) for kind in KINDS]      # in flight ...
        gpu.upload(scene_loader("scene_file_cube"), 32, 32)           # ... while the scene they read is replaced
    for kind, res in zip(KINDS, got):
        assert_same(host_results(res), ref[kind], f"re-upload {kind}")


# ---- 5. refusals, before anything is enqueued ------------------------------------------------------------------------------------
def query(kind, n, o=None, d=None, found=None, index=None, t=None, size=None):
    q = api.RayQuery()
    q.struct_size = C.sizeof(api.RayQuery) if size is None else size
    q.kind, q.n = kind, n
    q.origins, q.directions, q.found, q.index, q.tclosest = o, d, found, index, t
    return q


def rc(gpu, q):
    return gpu.L.ct_gpu_trace_rays(gpu.device, None if q is None else C.byref(q))


@pytest.mark.gpu
def test_refusals(scene_loader, gpu):
    import torch
    fs = scene_loader("scene_file_cube")
    gpu.upload(fs, 32, 32)
    n = 64
    rng = np.random.default_rng(9)
    o, d = stack(ray_families(fs, rng, scale=0.1))
    o, d = o[:n], d[:n]
    ot, dt = torch_rays(o, d)
    out = torch.zeros(n + 1, dtype=torch.int32, device="cuda:0")
    good = dict(o=ot.data_ptr(), d=dt.data_ptr(), found=out.data_ptr())
    assert rc(gpu, query(0, n, **good)) == 0
    host_o = np.ascontiguousarray(o)
    pinned = torch.from_numpy(host_o).pin_memory()
    for bad in (dict(good, o=host_o.ctypes.data), dict(good, d=pinned.data_ptr()), dict(good, found=np.zeros(n, np.uint32).ctypes.data),
                dict(good, o=ot.data_ptr() + 4), dict(good, found=out.data_ptr() + 2), dict(good, o=None), dict(good, d=None)):
        assert rc(gpu, query(0, n, **bad)) == CT_ERR_INVALID, bad
    assert rc(gpu, query(3, n, **good)) == CT_ERR_INVALID
    assert rc(gpu, query(-1, n, **good)) == CT_ERR_INVALID
    assert rc(gpu, query(0, n, size=C.sizeof(api.RayQuery) - 8, **good)) == CT_ERR_INVALID
    assert rc(gpu, None) == CT_ERR_INVALID
    assert rc(gpu, query(0, 1 << 31, **good)) == CT_ERR_LIMIT
    if torch.cuda.device_count() > 1:
        other = ot.to("cuda:1")
        assert rc(gpu, query(0, n, **dict(good, o=other.data_ptr()))) == CT_ERR_INVALID
    # accepted: n = 0 with no arrays, NULL outputs
    assert rc(gpu, query(1, 0)) == 0
    assert rc(gpu, query(2, n, o=ot.data_ptr(), d=dt.data_ptr())) == 0
    torch.cuda.synchronize()
    assert int(out[n]) == 0                                          # nothing written past n
    for bad in (ot.float(), torch.zeros((n, 6), dtype=torch.float64, device="cuda:0")[:, ::2]):        # float32, not contiguous
        with pytest.raises(ValueError):
            gpu.trace_rays(bad, dt)
    gpu.shutdown()
    assert rc(gpu, query(0, n, **good)) == CT_ERR_NO_SCENE


def test_python_refuses_host_tensors_and_unknown_kinds():
    torch = pytest.importorskip("torch")
    if not os.path.exists(api.GPU_LIB):
        pytest.skip("libct_gpu.so not built")
    r = ct.GpuRenderer(0)
    o = torch.zeros((4, 3), dtype=torch.float64)
    for bad in (o, o.float(), o.numpy().tolist()):
        with pytest.raises(ValueError):
            r.trace_rays(bad, o)
    with pytest.raises(ValueError):
        r.trace_rays(o, o, "ambient")
