"""The early-exit walks ray by ray (ct_gpu_debug_early: the path k_shadow's and k_bounce's rays take -- the walk, parking,
k_overflow, k_overflow_huge) against the oracle, on the bundled scenes and on caller trees at the ABI's limits: depth 96
(kStackMax), wide-walk stacks that overflow, a tree that is not nested, and trees whose leaf positions do not increase along
the reference's DFS.  Every answer must equal the oracle's bit for bit: `found` of a shadow ray (ray.t = 1e30f), `index` of a
reflection ray (ray.t = 0, the first barycentric pass in DFS order)."""
import contextlib
import dataclasses

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import host
from cobbletrace_b200.sceneio import FlatScene, LT_AMBIENT, LT_POINT, LT_DIRECTIONAL
from oracle import ct_oracle_py as O

pytestmark = pytest.mark.gpu

DBG = ct.CT_FLAG_KEEP_HITS | ct.CT_FLAG_COUNT_TESTS
FINF = 4294967296.0                                     # raythread.cpp:58: a reflection "miss" puts the shading point this far out
WALKED, OVERFLOW, HUGE, IN_PLACE = 0, 1, 2, 3          # ct_gpu_debug_early's path codes
OPTION_NAMES = ("traversal_budget", "overflow_warp_budget", "any_leaves", "primary_budget", "primary_split")
OPTIONS = {
    "default": {},
    "budget6": {"traversal_budget": 6},                                     # nearly every ray goes through k_overflow
    "budget6_warp1": {"traversal_budget": 6, "overflow_warp_budget": 1},    # ... and on to k_overflow_huge
    "unlimited": {"traversal_budget": 1 << 30},                             # only a full stack parks a ray
    "leaves5": {"any_leaves": 5},
    "leaves12": {"any_leaves": 12},
    "leaves64": {"any_leaves": 64},
}


@contextlib.contextmanager
def options(**kw):
    try:
        for k, v in kw.items():
            ct.api.set_option(k, v)
        yield
    finally:
        for k in OPTION_NAMES:
            ct.api.set_option(k, 0)


@pytest.fixture
def gpu():
    r = ct.GpuRenderer(0)
    yield r
    r.shutdown()


# ---- scenes ------------------------------------------------------------------------------------------------------------
def _lights_and_camera(cam_pos=(0.0, 0.0, 0.0)):
    return dict(light_type=np.array([LT_AMBIENT, LT_POINT, LT_DIRECTIONAL], np.int32), light_intensity=np.array([0.2, 0.6, 0.3], np.float32),
                light_pos=np.array([[0, 0, 0], [0.5, 0.3, -30.0], [0, 0, 0]]), light_dir=np.array([[0, 0, 0], [0, 0, 0], [0.2, 0.1, -1.0]]),
                cam_pos=np.array(cam_pos, np.float64), cam_rot=np.eye(3).reshape(9))


def _materials(rng, n, reflection):
    return dict(mat_color=rng.integers(0x202020, 0xffffff, n).astype(np.uint32), mat_specular=rng.choice(np.array([-1, 0, 10, 500], np.int32), n),
                mat_reflection=np.full(n, reflection, np.float32))


def soup(rng, n_tri=400, reflection=0.0):
    """Random triangle soup in front of a camera at the origin looking down +z, BVH from the host builder."""
    c = rng.normal(size=(n_tri, 3)) * 1.5 + np.array([0.0, 0.0, 6.0])
    a, b = rng.normal(size=(n_tri, 3)) * 0.6, rng.normal(size=(n_tri, 3)) * 0.6
    tri = np.concatenate([c - (a + b) / 3, c - (a + b) / 3 + a, c - (a + b) / 3 + b], 1)
    fs = FlatScene(tri=tri, **_materials(rng, n_tri, reflection), **_lights_and_camera())
    return host.HostScene.from_flat(fs).to_flat(with_bvh=True)


def flat_tree(tree, tri, rng, reflection=0.5, cam_pos=(0.0, 0.0, -20.0), nest=True):
    """A caller's tree as arrays.  `tree`: a leaf is a list of triangle ids, an interior node a tuple (left, right); children are
    stored next to each other (left_node, left_node + 1), leaves take positions in DFS order, every box is the exact union of its
    node's triangles (a nested tree) -- or, nest=False, interior boxes other than the root's shrink by 2 % about their centre."""
    nodes = []                                          # [left, first, count, tris of the subtree]
    tri_index = []

    def alloc():
        nodes.append([0, 0, 0, None])
        return len(nodes) - 1

    def fill(node, i):
        if isinstance(node, list):
            nodes[i][1], nodes[i][2] = len(tri_index), len(node)
            tri_index.extend(node)
            nodes[i][3] = list(node)
            return nodes[i][3]
        l = alloc(); alloc()
        nodes[i][0] = l
        nodes[i][3] = fill(node[0], l) + fill(node[1], l + 1)
        return nodes[i][3]

    fill(tree, alloc())
    n = len(nodes)
    v = tri.reshape(-1, 3, 3)
    nmin = np.array([v[nd[3]].reshape(-1, 3).min(0) for nd in nodes]); nmax = np.array([v[nd[3]].reshape(-1, 3).max(0) for nd in nodes])
    if not nest:
        inner = np.array([i for i in range(1, n) if nodes[i][2] == 0], np.int64)
        mid = 0.5 * (nmin[inner] + nmax[inner])
        nmin[inner] = mid + 0.98 * (nmin[inner] - mid); nmax[inner] = mid + 0.98 * (nmax[inner] - mid)
    fs = FlatScene(tri=tri, **_materials(rng, tri.shape[0], reflection), **_lights_and_camera(cam_pos),
                   node_min=nmin, node_max=nmax, node_left=np.array([nd[0] for nd in nodes], np.uint32),
                   node_first=np.array([nd[1] for nd in nodes], np.uint32), node_count=np.array([nd[2] for nd in nodes], np.uint32),
                   tri_index=np.array(tri_index, np.uint32))
    return fs


def tree_depth(fs):
    """Depth of the reference's DFS (the root counts 1), as ct_gpu_upload_scene measures it."""
    best, st = 0, [(0, 1)]
    while st:
        i, d = st.pop()
        best = max(best, d)
        if fs.node_count[i] == 0:
            st += [(int(fs.node_left[i]), d + 1), (int(fs.node_left[i]) + 1, d + 1)]
    return best


def dfs_leaves(fs):
    out, st = [], [0]
    while st:
        i = st.pop()
        if fs.node_count[i] > 0:
            out.append(i)
        else:
            st += [int(fs.node_left[i]) + 1, int(fs.node_left[i])]        # left popped first: the reference's order
    return out


def reverse_leaf_order(fs):
    """The same tree -- boxes, and triangles per leaf -- with the leaves' triangle ranges renumbered in reverse DFS order."""
    first, index, pos = fs.node_first.copy(), np.zeros_like(fs.tri_index), 0
    for leaf in reversed(dfs_leaves(fs)):
        a, c = int(fs.node_first[leaf]), int(fs.node_count[leaf])
        first[leaf] = pos
        index[pos:pos + c] = fs.tri_index[a:a + c]
        pos += c
    return dataclasses.replace(fs, node_first=first, tri_index=index)


def decoy(rng, k):
    """A sliver whose box holds the z axis (and the origin) but whose plane crosses the axis outside the triangle: its projection
    lies in x + y <= -0.7, the axis at x + y = 0."""
    a = 0.05 + 0.5 * rng.random()
    zs = rng.uniform(-5.0, -4.0), rng.uniform(4.0, 5.0)
    return np.array([-1.0 - a, 0.1, zs[0], 0.1, -1.0 - a, zs[1], -0.85, 0.15, 0.01 * k - 0.3])


def target():
    """A triangle across the axis (the DFS-last leaf: the first triangle an axis ray meets)."""
    return np.array([-2.0, -2.0, -0.5, 3.0, -2.0, 0.5, -2.0, 3.0, 0.25])


def comb(levels, rng):
    """levels interior nodes, each (interior, leaf): depth levels + 1.  The closest-hit walk pushes every right (leaf) child."""
    tri = np.array([decoy(rng, k) for k in range(levels)] + [target()])
    node = ([levels - 1], [levels])                     # the deepest pair: two leaves
    for k in range(levels - 2, -1, -1):
        node = (node, [k])
    return flat_tree(node, tri, rng)


def spine(rng, nest=True):
    """A spine of depth 96 (left children) whose right children are interior nodes over two interior nodes of two leaves each,
    all of them decoys but the DFS-last leaf: an any-hit walk along the axis passes every box, meets no triangle before that
    leaf and pushes three wide children per wide level on the way down -- kWideStack overflows."""
    tri, levels = [], 93
    def leaf(t=None):
        tri.append(decoy(rng, len(tri)) if t is None else t)
        return [len(tri) - 1]
    subtree = lambda last=None: ((leaf(), leaf()), (leaf(), leaf(last)))
    hang = [subtree(target())] + [subtree() for _ in range(levels)]
    node = (hang[-1], hang[-2])
    for k in range(levels - 2, -1, -1):
        node = (node, hang[k])
    fs = flat_tree(node, np.array(tri), rng, nest=nest)
    assert tree_depth(fs) == 96
    return fs


def geometric(rng, n=97):
    """Triangles whose centroids form a geometric series along x (ratio 0.45, sizes shrinking with them): BuildBVH's midpoint
    split peels one triangle off per level, a comb of depth about n built by the product's own builder."""
    c = 0.45 ** np.arange(n)
    s = 0.1 * c
    tri = np.stack([c - s, -s, -s, c + s, s, -s, c, -s, s], 1)
    fs = FlatScene(tri=tri, **_materials(rng, n, 0.5), **_lights_and_camera((0.5, 0.0, -2.0)))
    return host.HostScene.from_flat(fs).to_flat(with_bvh=True)


# ---- ray families --------------------------------------------------------------------------------------------------------
def surface_points(fs, rng, n):
    k = rng.integers(0, fs.n_tri, n)
    w = rng.dirichlet([1, 1, 1], n)
    return (fs.tri[k].reshape(-1, 3, 3) * w[:, :, None]).sum(1), k


def ray_families(fs, rng, scale=1.0):
    """{family: (origins, directions)}, seeded; `scale` thins them out."""
    m = lambda x: max(4, int(x * scale))
    fam = {}
    lights = [np.asarray(p) for t, p, d in zip(fs.light_type, fs.light_pos, fs.light_dir) if t == LT_POINT]
    dirs = [np.asarray(d) for t, p, d in zip(fs.light_type, fs.light_pos, fs.light_dir) if t == LT_DIRECTIONAL]
    o, _ = surface_points(fs, rng, m(600))
    if lights or dirs:
        aim = [lights[i] - o[j] if i < len(lights) else dirs[i - len(lights)] for j, i in enumerate(rng.integers(0, len(lights) + len(dirs), len(o)))]
        fam["surface->light"] = (o, np.array(aim))
    o, _ = surface_points(fs, rng, m(600))
    p, _ = surface_points(fs, rng, len(o))
    fam["surface->point"] = (o, (p - o) * rng.uniform(0.3, 3.0, (len(o), 1)))
    # occluders at t just beyond and just inside 1e-4 |d| (bvh.cpp:152): a point X on a triangle, the origin 1e-4 (1 + e) d before it
    x, _ = surface_points(fs, rng, m(300))
    d = rng.normal(size=x.shape)
    e = rng.choice(np.array([-1e-2, -1e-4, -1e-6, 1e-6, 1e-4, 1e-2]), (len(x), 1))
    fam["t=1e-4"] = (x - 1e-4 * (1 + e) * d, d)
    # one or two zero direction components (the binary walk: no conservative tests)
    o, _ = surface_points(fs, rng, m(400))
    p, _ = surface_points(fs, rng, len(o))
    d = p - o + rng.normal(size=o.shape) * 0.1
    zero = rng.integers(0, 3, len(o))
    d[np.arange(len(o)), zero] = 0.0
    two = rng.random(len(o)) < 0.3
    d[np.flatnonzero(two), (zero[two] + 1) % 3] = 0.0
    fam["zero component"] = (o, d)
    # the shading point of a reflection "miss": FINF ray lengths out (every box passes)
    o, _ = surface_points(fs, rng, m(48))
    d = rng.normal(size=o.shape)
    far = o + FINF * d
    aim = np.array([(lights[0] - f) if lights else -dd for f, dd in zip(far, d)])
    pick = rng.integers(0, 3, (len(o), 1))                            # at a light; straight back (every box passes); nearly back
    fam["far origin"] = (far, np.where(pick == 0, aim, np.where(pick == 1, -d, -d + rng.normal(size=d.shape) * 0.3)))
    # in the plane of a box face of the uploaded tree, along its edges, from its corners
    k = rng.integers(0, fs.n_nodes, m(400))
    lo, hi = fs.node_min[k], fs.node_max[k]
    ax = rng.integers(0, 3, len(k))
    side = rng.random(len(k)) < 0.5
    o = lo + (hi - lo) * rng.uniform(-0.2, 1.2, lo.shape)
    ar = np.arange(len(k))
    o[ar, ax] = np.where(side, lo[ar, ax], hi[ar, ax])
    d = rng.normal(size=o.shape)
    d[ar, ax] = 0.0
    e = np.flatnonzero(rng.random(len(k)) < 0.4)                      # ... along an edge: a second coordinate on a face, a second zero
    ax2 = (ax[e] + 1) % 3
    o[e, ax2] = np.where(side[e], hi[e, ax2], lo[e, ax2])
    d[e, ax2] = 0.0
    fam["box face/edge"] = (o, d)
    k = rng.integers(0, fs.n_nodes, m(200))
    corner = np.where(rng.random((len(k), 3)) < 0.5, fs.node_min[k], fs.node_max[k])
    d = np.round(rng.normal(size=corner.shape) * 8) / 8 + 0.0625      # dyadic: corner - 2 d is exact, the line runs through the corner
    fam["box corner"] = (np.concatenate([corner, corner - 2 * d]), np.concatenate([rng.normal(size=d.shape), d]))
    # along (and across) edges shared by triangles of different leaves
    leaf_of = np.zeros(fs.n_tri, np.int64)
    for leaf in np.flatnonzero(fs.node_count > 0):
        leaf_of[fs.tri_index[fs.node_first[leaf]:fs.node_first[leaf] + fs.node_count[leaf]]] = leaf
    v = fs.tri.reshape(-1, 3, 3)
    owner = {}
    shared = []
    for t in range(fs.n_tri):
        for a, b in ((0, 1), (1, 2), (2, 0)):
            key = tuple(sorted((tuple(v[t, a]), tuple(v[t, b]))))
            u = owner.setdefault(key, t)
            if u != t and leaf_of[u] != leaf_of[t]:
                shared.append(key)
    if shared:
        pick = [shared[i] for i in rng.integers(0, len(shared), m(300))]
        a = np.array([p[0] for p in pick]); b = np.array([p[1] for p in pick])
        along = rng.random((len(a), 1)) < 0.5
        mid = a + (b - a) * rng.uniform(0, 1, (len(a), 1))
        off = rng.normal(size=a.shape)
        fam["shared edge"] = (np.where(along, a - (b - a), mid + off), np.where(along, b - a, -off))
    return fam


def axis_rays(rng, n=200):
    """Down the spine: the origin at (0, 0, -10) / inside every box (the origin), directions near +z."""
    d = np.column_stack([rng.normal(size=(n, 2)) * 0.02, np.ones(n)])
    d[:8, :2] = 0.0
    o = np.zeros((n, 3))
    o[: n // 2, 2] = -10.0
    return {"spine axis": (o, d)}


def stack(fam):
    return np.concatenate([f[0] for f in fam.values()]), np.concatenate([f[1] for f in fam.values()])


def oracle_early(fs, fam):
    """The oracle's answers for both modes: (found, index) of ClosestIntersection with ray.t = 1e30f and with ray.t = 0."""
    osc = O.OracleScene(fs)
    o, d = stack(fam)
    return {mode: osc.closest_many(o, d, 1e30 if mode == 0 else 0.0)[:2] for mode in (0, 1)}


def check_early(gpu, ref, fam, what, mode, opt):
    """debug_early on every family against the oracle's answers; returns the path codes by family."""
    o, d = stack(fam)
    tag = np.concatenate([[name] * len(f[0]) for name, f in fam.items()])
    found, index, path = gpu.debug_early(o, d, mode)
    rfound, rindex = ref[mode]
    bad = (found != rfound) if mode == 0 else (index != rindex) | (found != 1)
    if bad.any():
        i = np.flatnonzero(bad)
        names, counts = np.unique(tag[i], return_counts=True)
        raise AssertionError(f"{what} {opt} mode {mode}: {len(i)} of {len(o)} rays differ from the oracle "
                             f"({dict(zip(names, counts.tolist()))}); first: ray {i[0]} {tag[i[0]]} gpu {found[i[0]], index[i[0]], path[i[0]]}, "
                             f"oracle {rfound[i[0]], rindex[i[0]]}")
    return {name: path[tag == name] for name in fam}


def run_matrix(gpu, fs, fam, what, W=32, H=32):
    """Both modes under every option setting; returns {(option, mode): {family: path codes}}."""
    ref = oracle_early(fs, fam)
    out = {}
    for opt, kw in OPTIONS.items():
        with options(**kw):
            gpu.upload(fs, W, H, max_depth=2)
            for mode in (0, 1):
                out[opt, mode] = check_early(gpu, ref, fam, what, mode, opt)
    return out


def n_path(paths, code, families=None):
    return sum(int((p == code).sum()) for name, p in paths.items() if families is None or name in families)


# ---- bundled scenes and a soup -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["scene_import_bunny", "pc_big", "scene_file_cube", "soup"])
def test_early_walks_ray_by_ray(name, scene_loader, gpu):
    rng = np.random.default_rng(sum(map(ord, name)))
    fs = soup(rng) if name == "soup" else scene_loader(name)
    fam = ray_families(fs, rng, scale=0.5 if name == "scene_import_bunny" else 1.0)
    res = run_matrix(gpu, fs, fam, name)
    for mode in (0, 1):
        assert n_path(res["budget6", mode], OVERFLOW) > 50, (name, mode)
        assert n_path(res["budget6_warp1", mode], HUGE) > 50, (name, mode)
        for p in res["unlimited", mode].values():                    # nothing but a full stack (or an origin FINF away) parks
            assert np.isin(p, [WALKED, IN_PLACE]).all(), (name, mode)
    # shadow rays from FINF away that reach the root are parked at once: k_overflow_huge, or in place when the scene is too small
    # to park anything (node and triangle counts below the default budget); the others miss the root box
    far = res["default", 0]["far origin"]
    at_once = HUGE if fs.n_nodes + fs.n_tri > 384 else IN_PLACE
    assert np.isin(far, [WALKED, at_once]).all() and (far == at_once).any(), (name, far)


# ---- caller trees at the limits ------------------------------------------------------------------------------------------------
def check_closest(gpu, fs, fam, what):
    osc = O.OracleScene(fs)
    o = np.concatenate([f[0] for f in fam.values()]); d = np.concatenate([f[1] for f in fam.values()])
    for t0 in (1e30, 0.0):
        found, index, t = gpu.debug_closest(o, d, t0)
        rf, ri, rt = osc.closest_many(o, d, t0)
        assert np.array_equal(found, rf) and np.array_equal(index, ri) and np.array_equal(t.view(np.uint32), rt.view(np.uint32)), (what, t0)


def check_frame(gpu, fs, what, W=48, H=48, depth=3, **kw):
    oframe, ohits, _ = O.OracleScene(fs).render(W, H, max_depth=depth)
    with options(**kw):
        gpu.upload(fs, W, H, max_depth=depth, flags=DBG)
        gpu.render_tile()
    frame = gpu.readback()
    found, index, t = gpu.readback_hits()
    traced = ohits["found"] != 0xFFFFFFFF
    assert np.array_equal(frame, oframe), f"{what} {kw}: {int((frame != oframe).sum())} pixels differ"
    assert np.array_equal(found, ohits["found"]) and np.array_equal(index[traced], ohits["index"][traced]), (what, kw)
    assert np.array_equal(t[traced].view(np.uint32), ohits["t"][traced].view(np.uint32)), (what, kw)
    return oframe


PARK_ALL = dict(primary_budget=1, primary_split=1, traversal_budget=6)


def check_tree(gpu, fs, rng, what):
    fam = {**axis_rays(rng), **ray_families(fs, rng, scale=0.3)}
    res = run_matrix(gpu, fs, fam, what)
    gpu.upload(fs, 32, 32)
    check_closest(gpu, fs, fam, what)
    for kw in ({}, PARK_ALL):
        check_frame(gpu, fs, what, **kw)
    return res


def test_comb_of_depth_96_and_97(gpu):
    rng = np.random.default_rng(96)
    fs = comb(95, rng)
    assert tree_depth(fs) == 96
    res = check_tree(gpu, fs, rng, "comb 96")
    # first-line walks from inside every box push two leaves per wide level: the wide stack fills and the ray is parked (in place:
    # the tree is too small for parking buffers at the default budget)
    assert n_path(res["unlimited", 1], IN_PLACE, ["spine axis"]) > 0
    assert n_path(res["default", 1], IN_PLACE, ["spine axis"]) > 0
    deep = comb(96, rng)
    assert tree_depth(deep) == 97
    gpu.upload(fs, 48, 48, max_depth=3)
    gpu.render_tile()
    before = gpu.readback()
    with pytest.raises(ct.CtError) as e:
        gpu.upload(deep, 48, 48, max_depth=3)
    assert e.value.code == -5                                    # CT_ERR_LIMIT
    gpu.render_tile()                                            # the scene uploaded before is still there and renders the same
    assert np.array_equal(gpu.readback(), before)
    check_frame(gpu, fs, "comb 96 after a refused upload")


@pytest.mark.parametrize("nest", [True, False])
def test_spine_overflows_the_wide_stack(nest, gpu):
    rng = np.random.default_rng(7 + nest)
    fs = spine(rng, nest=nest)
    res = check_tree(gpu, fs, rng, f"spine nest={nest}")
    if nest:
        # an any-hit walk down the axis meets no triangle before the DFS-last leaf and pushes three wide children per level
        assert n_path(res["unlimited", 0], IN_PLACE, ["spine axis"]) > 0
        assert n_path(res["default", 0], OVERFLOW, ["spine axis"]) > 0
    else:
        # not nested: the exact binary walks, at full depth, in the rays' own threads
        assert n_path(res["unlimited", 0], IN_PLACE, ["spine axis"]) == 0


def test_host_builder_comb_from_a_geometric_series(gpu):
    rng = np.random.default_rng(45)
    fs = geometric(rng)
    ref = O.build_bvh(fs.tri)
    assert all(np.array_equal(getattr(fs, k), ref[k]) for k in ref), "host BuildBVH differs from the oracle's"
    depth = tree_depth(fs)
    assert 90 <= depth <= 96, depth
    rng2 = np.random.default_rng(46)
    d = np.column_stack([np.ones(200), rng2.normal(size=(200, 2)) * 0.01])
    o = np.tile([-3.0, 0.0, 0.0], (200, 1))
    o[100:] = [1e-20, 0.0, 0.0]                                  # inside the deepest boxes
    fam = {"along x": (o, d), **ray_families(fs, rng2, scale=0.2)}
    run_matrix(gpu, fs, fam, "geometric")
    gpu.upload(fs, 32, 32)
    check_closest(gpu, fs, fam, "geometric")
    for kw in ({}, PARK_ALL):
        check_frame(gpu, fs, "geometric", **kw)


# ---- leaves out of DFS order ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["scene_import_bunny", "soup"])
def test_leaves_out_of_dfs_order(name, scene_loader, gpu):
    """A caller's tree whose leaf positions run against the DFS: reflection rays must still take the DFS-first pass when
    they are parked (k_overflow's minimum over lanes, k_overflow_huge's atomicMin)."""
    rng = np.random.default_rng(11)
    fs = (soup(rng, 600) if name == "soup" else scene_loader(name)).with_reflection(0.5)
    rev = reverse_leaf_order(fs)
    assert not np.array_equal(rev.node_first, fs.node_first)
    W, H = (96, 96) if name == "soup" else (128, 128)
    ref = check_frame(gpu, rev, f"{name} reversed", W, H, depth=2)                # no parking: checks the test itself
    assert np.array_equal(ref, O.OracleScene(fs).render(W, H, max_depth=2, want_hits=False)[0])      # same tree, same picture
    for kw in ({"traversal_budget": 6}, {"traversal_budget": 6, "overflow_warp_budget": 1}):
        check_frame(gpu, rev, f"{name} reversed", W, H, depth=2, **kw)
    o, _ = surface_points(rev, rng, 3000)
    fam = {"surface": (o, rng.normal(size=o.shape))}
    ref = oracle_early(rev, fam)
    for opt in ("default", "budget6", "budget6_warp1"):
        with options(**OPTIONS[opt]):
            gpu.upload(rev, 32, 32, max_depth=2)
            check_early(gpu, ref, fam, f"{name} reversed", 1, opt)


def test_tie_in_t_between_sibling_leaves_out_of_dfs_order(gpu):
    """Coincident duplicate triangles in sibling leaves, with different colours: the reference keeps the DFS-first one (its
    t is not below the other's, bvh.cpp:212).  Primary rays parked for k_primary_split must do the same (its replay orders the
    candidates by leaf position; a small traversal_budget lets a tree this small park at all)."""
    rng = np.random.default_rng(5)
    big = np.array([-4.0, -4.0, 6.0, 5.0, -3.0, 6.5, -3.0, 5.0, 5.5])
    far = np.array([-4.0, -4.0, 9.0, 5.0, -3.0, 9.5, -3.0, 5.0, 9.0])
    tri = np.array([big, big, far, decoy(rng, 0) + np.array([0, 0, 7.0] * 3)])
    fs = flat_tree((([0], [1]), ([2], [3])), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0))
    fs = dataclasses.replace(fs, mat_color=np.array([0x2040e0, 0xe04020, 0x20e040, 0x808080], np.uint32))
    for tree in (fs, reverse_leaf_order(fs)):
        a = check_frame(gpu, tree, "tie", 48, 48, depth=0)
        b = check_frame(gpu, tree, "tie parked", 48, 48, depth=0, **PARK_ALL)
        assert np.array_equal(a, b)
    assert (a == O.OracleScene(fs).render(48, 48, max_depth=0, want_hits=False)[0]).all()
