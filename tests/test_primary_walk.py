"""Primary rays ray by ray (ct_gpu_debug_primary: the path a frame's primary rays take -- k_primary's budgeted walk, parking, the
real k_primary_long or the order-free k_primary_split, or the walk again in place when the parking buffer is full) against the
oracle.  found, index and the bits of tclosest must equal ClosestIntersection's with ray.t = 1e30f, under every primary_budget /
primary_split setting, on the bundled scenes and on caller trees built to reach each of k_primary_split's outcomes: decided by its
frontier and replay, or handed to the ordered walk for one of seven reasons."""
import ctypes as C

import numpy as np
import pytest

from oracle import ct_oracle_py as O
from cobbletrace_b200.sceneio import FlatScene
from test_walk_limits import (FINF, _lights_and_camera, _materials, decoy, flat_tree, gpu, options, ray_families,  # noqa: F401 (gpu: fixture)
                              reverse_leaf_order, soup, surface_points, target)

pytestmark = pytest.mark.gpu

OWN, LONG, SPLIT, IN_PLACE = 0, 1, 2, 3                  # path & 0xff
DECIDED, NO_SIGMA, NOT_NESTED, T_FINF, CAND_FULL, STACK_FULL, LATE, MANY = range(8)     # path >> 8 of a SPLIT ray
SPLIT_SETTINGS = {"split1": dict(primary_budget=1, primary_split=1), "split6": dict(primary_budget=6, primary_split=1),
                  "split40": dict(primary_budget=40, primary_split=1)}
SETTINGS = {"default": ({}, 0), "long1": (dict(primary_budget=1), 0),
            **{k: (v, 0) for k, v in SPLIT_SETTINGS.items()}, **{k + "_cap3": (v, 3) for k, v in SPLIT_SETTINGS.items()}}
SMALL_TREE = dict(traversal_budget=6)                  # a caller tree this small parks at all only with a small traversal budget


def stack(fam):
    return np.concatenate([f[0] for f in fam.values()]), np.concatenate([f[1] for f in fam.values()])


def run(gpu, fs, fam, what, extra=None, settings=SETTINGS, parked=SPLIT):
    """debug_primary under every setting against the oracle; {setting: {family: path codes}}.  parked: where primary_split sends the
    parked rays (SPLIT, or LONG on a tree whose leaf positions do not increase along the DFS)."""
    o, d = stack(fam)
    tag = np.concatenate([[name] * len(f[0]) for name, f in fam.items()])
    rf, ri, rt = O.OracleScene(fs).closest_many(o, d, 1e30)
    out, n_over = {}, {}
    for name, (kw, cap) in settings.items():
        with options(**{**(extra or {}), **kw}):
            gpu.upload(fs, 32, 32)
            found, index, t, path = gpu.debug_primary(o, d, cap)
        bad = (found != rf) | (index != ri) | (t.view(np.uint32) != rt.view(np.uint32))
        if bad.any():
            i = np.flatnonzero(bad)
            names, counts = np.unique(tag[i], return_counts=True)
            raise AssertionError(f"{what} {name}: {len(i)} of {len(o)} rays differ from the oracle ({dict(zip(names, counts.tolist()))}); "
                                 f"first: ray {i[0]} {tag[i[0]]} o={o[i[0]].tolist()} d={d[i[0]].tolist()} gpu {found[i[0]], index[i[0]], t[i[0]]} "
                                 f"path {path[i[0]] & 0xff}/{path[i[0]] >> 8}, oracle {rf[i[0]], ri[i[0]], rt[i[0]]}")
        out[name] = {f: path[tag == f] for f in fam}
        low = path & 0xff
        if name == "default":
            assert (low == OWN).all(), (what, name)
        elif name == "long1":
            assert np.isin(low, [OWN, LONG]).all(), (what, name)
            if (fs.node_count[fs.node_left[0]:fs.node_left[0] + 2] == 0).all():     # both root children interior: a hit takes 2 pair visits
                assert (low[rf == 1] == LONG).all(), (what, name)
        else:
            assert np.isin(low, [OWN, parked, IN_PLACE] if cap else [OWN, parked]).all(), (what, name)
            over = int((low != OWN).sum())                   # the budgeted walk alone decides which rays go over the budget
            if cap:                                          # ... of which the first `cap` are parked, the others walked in place
                base = n_over[name[:-len("_cap3")]]
                assert over == base and (low == IN_PLACE).sum() == max(0, base - cap), (what, name, base)
            n_over[name] = over
    return out


def outcomes(res, family):
    """k_primary_split's outcome codes over the split settings without a parking cap, for one family."""
    p = np.concatenate([res[k][family] for k in SPLIT_SETTINGS])
    return set((p[(p & 0xff) == SPLIT] >> 8).tolist())


def decided_share(res, families):
    p = np.concatenate([res[k][f] for k in SPLIT_SETTINGS for f in families])
    p = p[(p & 0xff) == SPLIT]
    return float(((p >> 8) == DECIDED).mean()) if len(p) else 0.0


def balanced(leaves):
    """Nested tuples over a list of leaves (lists of triangle ids), halving: leaves take positions in list order."""
    if len(leaves) == 1:
        return leaves[0]
    h = (len(leaves) + 1) // 2
    return (balanced(leaves[:h]), balanced(leaves[h:]))


def intersect(o, d, tri):
    """The oracle's IntersectTriangle (bvh.cpp:147-163) from ray.t = 1e30f: the t it would leave, or inf without a pass that lowers it."""
    L = O.lib()
    o = np.ascontiguousarray(o, np.float64); d = np.ascontiguousarray(d, np.float64); tri = np.ascontiguousarray(tri, np.float64)
    t = C.c_float(1e30)
    hit = L.ct_oracle_intersect_triangle(O._ptr(o), O._ptr(d), C.byref(t), O._ptr(tri))
    return t.value if hit and t.value < np.float32(1e30) else np.inf


def least_t_differs(fs, o, d):
    """Rays whose reference answer is NOT the triangle with the least t: an earlier leaf's triangle lowered ray.t below the rounded
    tmin of the leaf that holds the nearer one (brute force over every triangle with the oracle's IntersectTriangle)."""
    _, _, rt = O.OracleScene(fs).closest_many(o, d, 1e30)
    least = np.array([min(intersect(o[i], d[i], tr) for tr in fs.tri) for i in range(len(o))], np.float32)
    return rt > least


# ---- scenes ------------------------------------------------------------------------------------------------------------
def layer(z, half=2.0, rot=None, scale=1.0):
    """A square of side 2 half at height z, as two triangles sharing the diagonal (x = y); rot: a 3x3 rotation about the origin."""
    q = np.array([[-half, -half, z], [half, -half, z], [half, half, z], [-half, half, z]]) * scale
    if rot is not None:
        q = q @ rot.T
    return [np.concatenate([q[0], q[1], q[2]]), np.concatenate([q[0], q[2], q[3]])]


def rotation(rng):
    a = rng.normal(size=(3, 3))
    q, _ = np.linalg.qr(a)
    return q


def stack_scene(rng, K, ulps, per_leaf, order, oblique=False, scale=1.0):
    """K parallel squares (2 triangles each) `ulps` float ulps apart at z = 6 (ulp 2^-21), axis-aligned -- zero-thickness leaf
    boxes -- or rotated; per_leaf triangles to a leaf; order: leaf (DFS) order against t order ("same", "reversed", "shuffled")."""
    rot = rotation(rng) if oblique else None
    tri = np.array([t for k in range(K) for t in layer(6.0 + k * ulps * 2.0 ** -21, rot=rot, scale=scale)])
    ids = np.arange(len(tri))
    if order == "reversed":
        ids = ids[::-1].copy()
    elif order == "shuffled":
        ids = rng.permutation(ids)
    leaves = [ids[i:i + per_leaf].tolist() for i in range(0, len(ids), per_leaf)]
    return flat_tree(balanced(leaves), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0)), rot


def stack_rays(rng, rot, n=120, scale=1.0):
    """Rays from z = 0 through the squares: interiors, the shared diagonal, vertices; normal, oblique and grazing."""
    pts = np.concatenate([rng.uniform(-1.9, 1.9, (n, 2)), np.repeat(rng.uniform(-1.9, 1.9, (n // 2, 1)), 2, 1),
                          np.array([[-2.0, -2.0], [2.0, -2.0], [2.0, 2.0], [-2.0, 2.0], [0.0, 0.0]] * 4)])
    m = len(pts)
    aim = np.column_stack([pts, np.full(m, 6.0)])
    kind = rng.integers(0, 4, m)
    normal = np.where(kind[:, None] == 0, [[0.0, 0.0, 1.0]], [[2.0 ** -30, -(2.0 ** -31), 1.0]])     # exactly, or with a slab filter
    d = np.where(kind[:, None] <= 1, normal, np.where(kind[:, None] == 2, np.column_stack([rng.normal(size=(m, 2)) * 0.3, np.ones(m)]),
                                                      np.column_stack([rng.normal(size=(m, 2)) * 3.0, np.full(m, 0.02)])))
    o = aim - 6.0 * d / d[:, 2:3]
    if rot is not None:
        o, d, aim = o @ rot.T, d @ rot.T, aim @ rot.T
    return o * scale, d


def fan(rng, n=64):
    """n thin triangles around the vertex (0, 0, 5), each in its own leaf of a balanced tree, tilted a little each."""
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    w = 2 * np.pi / n
    tri = np.array([[0, 0, 5.0, 3 * np.cos(a), 3 * np.sin(a), 5.0 + 0.2 * np.sin(3 * a), 3 * np.cos(a + w), 3 * np.sin(a + w), 5.0 + 0.2 * np.sin(3 * a)]
                    for a in ang])
    fs = flat_tree(balanced([[i] for i in range(n)]), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0))
    d = np.column_stack([rng.normal(size=(60, 2)) * 0.2, np.ones(60)])
    o = np.array([0.0, 0.0, 5.0]) - 5.0 * d                    # through the shared vertex (dyadic: exact)
    d[:8] = [0.0, 0.0, 1.0]; o[:8] = [0.0, 0.0, 0.0]
    return fs, {"fan vertex": (o, d)}


def duplicates(rng):
    """Exact duplicates of one triangle in one leaf, in sibling leaves and in cousin leaves; the tie goes to the DFS-first one."""
    t = np.array([-3.0, -3.0, 6.0, 4.0, -2.0, 6.5, -2.0, 4.0, 5.5])
    tri = np.array([t] * 6 + [decoy(rng, 0) + np.array([0, 0, 9.0] * 3), decoy(rng, 1) + np.array([0, 0, 9.0] * 3)])
    fs = flat_tree(((([0, 1], [2]), ([6], [3])), (([7], [4]), [5])), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0))
    w = rng.dirichlet([1, 1, 1], 200)
    p = w @ t.reshape(3, 3)
    d = np.column_stack([rng.normal(size=(200, 2)) * 0.3, np.ones(200)])
    return fs, {"duplicates": (p - 6.0 * d, d)}


def leaf_pair(rng, n=300):
    """One leaf holding two squares half a float ulp apart at z = 3, the farther one first.  The reference tests the leaf's box once,
    then both triangles: on rays where the farther triangle's float t is no more than the box's tmin and the nearer one's is lower,
    the nearer one wins although the box's tmin is not below the ray.t the farther one left.  A replay that tested the box again
    for every candidate would drop it.  Returns the scene, the rays and how many of them are of this kind."""
    far, near = layer(3.0 + 2.0 ** -23)[0], layer(3.0)[0]
    tri = np.array([far, near] + [decoy(rng, k) + np.array([0, 0, 20.0] * 3) for k in range(3)])
    fs = flat_tree((([0, 1], [2]), ([3], [4])), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0))
    x = rng.uniform(-1.5, 1.9, n)
    aim = np.column_stack([x, rng.uniform(-1.9, x - 0.05), np.full(n, 3.0)])        # inside both triangles (below the diagonal)
    d = np.column_stack([rng.normal(size=(n, 2)) * 0.4, rng.uniform(0.5, 1.0, n)])
    o = aim - rng.uniform(1.0, 10.0, (n, 1)) * d
    lo, hi = np.array([-2.0, -2.0, 3.0]), np.array([2.0, 2.0, 3.0 + 2.0 ** -23])
    n_kind = 0
    for i in range(n):
        t1, t2 = intersect(o[i], d[i], far), intersect(o[i], d[i], near)
        tmin = max(np.minimum(np.float32((lo - o[i]) / d[i]), np.float32((hi - o[i]) / d[i])))     # IntersectAABB's float tmin
        n_kind += bool(t2 < t1 <= tmin)
    return fs, {"leaf pair": (o, d)}, n_kind


def decoy_forest(rng, levels=18):
    """A complete tree of 2^levels leaves: decoy slivers whose boxes all hold the z axis, and a target in the DFS-last leaf.  Every
    conservative test along the axis accepts, so each round of the frontier takes 32 nodes off the warp's stack and pushes four
    children for each; the stack grows by about 96 entries per wide level and fills its 512 entries only on a tree this deep
    (9 wide levels; 4096 leaves peak at 256).  Stored in breadth-first order: node i has children 2i + 1, 2i + 2."""
    n = 1 << levels
    a = 0.05 + 0.5 * rng.random(n)
    z0, z1 = rng.uniform(-5.0, -4.0, n), rng.uniform(4.0, 5.0, n)
    k = np.arange(n) % 60
    tri = np.column_stack([-1.0 - a, np.full(n, 0.1), z0, np.full(n, 0.1), -1.0 - a, z1, np.full(n, -0.85), np.full(n, 0.15), 0.01 * k - 0.3])
    tri[-1] = target()
    v = tri.reshape(n, 3, 3)
    lo, hi = np.zeros((2 * n - 1, 3)), np.zeros((2 * n - 1, 3))
    lo[n - 1:], hi[n - 1:] = v.min(1), v.max(1)
    for lev in range(levels - 1, -1, -1):
        i = np.arange((1 << lev) - 1, (1 << (lev + 1)) - 1)
        lo[i] = np.minimum(lo[2 * i + 1], lo[2 * i + 2]); hi[i] = np.maximum(hi[2 * i + 1], hi[2 * i + 2])
    inner = np.arange(2 * n - 1) < n - 1
    fs = FlatScene(tri=tri, **_materials(rng, n, 0.0), **_lights_and_camera((0.0, 0.0, -10.0)), node_min=lo, node_max=hi,
                   node_left=np.where(inner, 2 * np.arange(2 * n - 1) + 1, 0).astype(np.uint32),
                   node_first=np.where(inner, 0, np.arange(2 * n - 1) - (n - 1)).astype(np.uint32),
                   node_count=np.where(inner, 0, 1).astype(np.uint32), tri_index=np.arange(n, dtype=np.uint32))
    d = np.column_stack([rng.normal(size=(40, 2)) * 1e-3, np.ones(40)])         # inside every decoy's box all the way
    o = np.tile([0.0, 0.0, -10.0], (40, 1))
    return fs, {"axis": (o, d)}


def outside_rays(fs, rng, n):
    """Rays from outside the scene's box at points on triangles."""
    p, _ = surface_points(fs, rng, n)
    lo, hi = fs.node_min[0], fs.node_max[0]
    u = rng.normal(size=p.shape)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    far = 2.0 * np.linalg.norm(hi - lo) + 1.0
    return p - far * u, u * rng.uniform(0.5, 2.0, (n, 1))


SCALES = (-40, -30, -20, 20, 40)


def with_scaled(fam, name):
    """The same rays with directions scaled by 2^k (exact): t, M and |a| of IntersectTriangle move with them."""
    o, d = fam[name]
    return {**fam, **{f"{name} 2^{k}": (o, d * 2.0 ** k) for k in SCALES}}


# ---- sigma at its limits -----------------------------------------------------------------------------------------------------
def sigma(bound, o, d):
    """tray_nearest_setup's sigma, for a ray whose largest term of M has a power-of-two direction component (float(d) and its
    float reciprocal exact)."""
    B = max(bound); O_ = np.abs(o).max(); D = np.abs(d).max()
    M = max((bound[k] + abs(o[k])) * abs(1.0 / d[k]) for k in range(3))
    if not (D * B * B <= 4096.0 and (O_ + B) * D * B <= 4096.0 and 2.0 ** -60 < M < 2.0 ** 60):
        return 0.0
    x = M * (2.0 ** -15 * 1.000001)
    f = np.float32(x)
    return float(f if f >= x else np.nextafter(f, np.float32(np.inf)))


def fadd_ru(a, b):
    x = float(a) + float(b)                              # exact in double
    f = np.float32(x)
    return float(f if f >= x else np.nextafter(f, np.float32(np.inf)))


def late_family(rng):
    """Two squares (A at z = 3, B about 1/8 ray lengths behind it) and rays (ox, oy, oz) + t (2^-10, 1/4, 0.8): sigma = 2^-15 M with
    M = (4 + ox) 2^10 (the x term: exact, as 2^-10 is) is just above 1/8, so B's triangle lies at the edge of the band t_A + sigma.
    With the reference's arithmetic, the rays kept are those where B's t is inside the band but the float tmin of B's flat leaf box
    is beyond it (IntersectTriangle's t rounds one ulp below the box's): the replay cannot tell from the leaf whether the reference
    enters it, and k_primary_split must give the ray up ("late")."""
    dz = 0.8
    zb = 3.0 + (0.125 + 6e-7) * dz
    tri = np.array(layer(3.0, half=4.0) + layer(zb, half=4.0) + [decoy(rng, 0) + np.array([0, 0, 20.0] * 3), decoy(rng, 1) + np.array([0, 0, 20.0] * 3)])
    fs = flat_tree((([0, 1], [2, 3]), ([4], [5])), tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0))
    bound = [max(abs(fs.node_min[:, k]).max(), abs(fs.node_max[:, k]).max()) for k in range(3)]
    d = np.array([2.0 ** -10, 0.25, dz])
    n = 20000
    o = np.column_stack([rng.uniform(0.0, 4e-5, n), rng.uniform(-1.0, 1.0, n), rng.uniform(-0.5, 0.5, n)])
    keep = []
    for i in range(n):
        ta = min(intersect(o[i], d, tri[0]), intersect(o[i], d, tri[1]))
        tb = min(intersect(o[i], d, tri[2]), intersect(o[i], d, tri[3]))
        s = sigma(bound, o[i], d)
        if not (np.isfinite(ta) and np.isfinite(tb) and s > 0):
            continue
        tmin_b = float(np.float32((zb - o[i, 2]) / dz))      # the z slab decides: the x / y slabs start far behind the origin
        if tb <= fadd_ru(ta, s) < tmin_b:
            keep.append(i)
        if len(keep) >= 40:
            break
    return fs, {"late": (o[keep], np.tile(d, (len(keep), 1)))}


def limit_rays(fs, rng):
    """Rays from the origin at the stack whose D B^2, (O + B) D B and M sit just inside / just outside tray_nearest_setup's limits.
    B = max bound.  With O = 0 the first two limits coincide (and (O + B) D B >= D B^2 always: D B^2 cannot be the only one
    broken); an origin O = B away breaks the second alone.  M is set by one small direction component (upper limit) or by
    all three large ones (lower limit, on a scene scaled to B = 2^-20)."""
    bnd = [max(abs(fs.node_min[:, k]).max(), abs(fs.node_max[:, k]).max()) for k in range(3)]
    B, bx = max(bnd), bnd[0]
    fam = {}
    base = np.array([0.125, 0.0625, 1.0])
    for side, f in (("in", 1 - 2 ** -8), ("out", 1 + 2 ** -8)):
        D = 4096.0 / B ** 2 * f                                 # O = 0: D B^2 = 4096 f
        o = np.zeros((30, 3))                                   # O = 0
        dd = np.tile(base / base.max() * D, (30, 1)) + np.column_stack([rng.uniform(-1, 1, (30, 2)) * 1e-3 * D, np.zeros(30)])
        fam[f"DB^2 {side}"] = (o, dd)
        D2 = 4096.0 / (2 * B * B) * f                           # O = B on the z axis: (O + B) D B = 4096 f, D B^2 = 2048 f
        o2 = np.tile([0.0, 0.0, -B], (30, 1))
        dd2 = np.tile(base / base.max() * D2, (30, 1)) + np.column_stack([rng.uniform(-1, 1, (30, 2)) * 1e-3 * D2, np.zeros(30)])
        fam[f"(O+B)DB {side}"] = (o2, dd2)
        dx = bx * 2.0 ** -60 / f                                # M = (bound_x + |o_x|) / |d_x| = 2^60 f
        o3 = np.zeros((30, 3))
        dd3 = np.column_stack([np.full(30, dx), rng.uniform(-0.2, 0.2, 30), np.ones(30)])
        fam[f"M high {side}"] = (o3, dd3)
    return fam


def lower_m_family(rng):
    """The lower limit of M on a stack scaled to B = 2^-20: every direction component about 2^40 (M = B / min |d_k| ~ 2^-60).  M
    bounds the t of every point in the scene's box, so below the limit no hit can lie beyond t = 1e-4: these rays find nothing,
    and inside the limit the frontier must say so itself."""
    fs, _ = stack_scene(rng, 4, 1, 1, "same", scale=2.0 ** -22)
    bx = max(abs(fs.node_min[:, 0]).max(), abs(fs.node_max[:, 0]).max())
    fam = {}
    for side, f in (("in", 1 + 2 ** -8), ("out", 1 - 2 ** -8)):
        s = bx / (2.0 ** -60 * f)                               # the x term is the largest: M = bound_x / s = 2^-60 f
        d = np.column_stack([np.full(40, s), np.full(40, s) * rng.uniform(1.0, 1.01, 40), np.full(40, 4.0 * s)])
        o = np.zeros((40, 3))
        fam[f"M low {side}"] = (o, d)
    return fs, fam


# ---- tests -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["scene_import_bunny", "pc_big", "scene_file_cube", "scene_import", "soup"])
def test_primary_walk_ray_by_ray(name, scene_loader, gpu):
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    fs = soup(rng) if name == "soup" else scene_loader(name)
    fam = ray_families(fs, rng, scale=0.25 if name == "scene_import_bunny" else 0.5)
    fam["outside"] = outside_rays(fs, rng, 300)
    fam = with_scaled(fam, "outside")
    res = run(gpu, fs, fam, name, SMALL_TREE if fs.n_nodes + fs.n_tri <= 384 else None)     # (scene_file_cube: 37 triangles)
    assert NO_SIGMA in outcomes(res, "outside 2^40") and NO_SIGMA in outcomes(res, "outside 2^20")
    assert NO_SIGMA not in outcomes(res, "outside 2^-20") and DECIDED in outcomes(res, "outside 2^-20")
    for f in fam:
        print(f"{name} {f}: split rays decided by the frontier {decided_share(res, [f]):.3f}, outcomes {sorted(outcomes(res, f))}")
    # Every split ray inside the rounding analysis was decided by the frontier on a B200 (share 1.000 on all five scenes); the share
    # of ALL split rays was 0.49 (bunny), 0.58 (pc_big), 0.69 (scene_import), 0.64 (soup): the others have sigma = 0 -- zero direction
    # components, origins 2^32 ray lengths out, the scaled directions and, on the bunny, D B^2 > 4096 for rays of length ~1 or more.
    p = np.concatenate([res[k][f] for k in SPLIT_SETTINGS for f in fam if " 2^" not in f])
    p = p[((p & 0xff) == SPLIT) & ((p >> 8) != NO_SIGMA)]
    assert len(p) > 10 and ((p >> 8) == DECIDED).mean() > 0.95, name
    # the call leaves a frame alone
    gpu.upload(fs, 64, 64, max_depth=2)
    gpu.render_tile()
    before = gpu.readback()
    o, d = stack(fam)
    with options(**SPLIT_SETTINGS["split6"]):
        gpu.debug_primary(o[:500], d[:500], 3)
    gpu.render_tile()
    assert np.array_equal(gpu.readback(), before)


STACKS = [(K, ulps, per_leaf, order, oblique) for K, ulps, per_leaf, order, oblique in [
    (2, 1, 1, "reversed", False), (4, 1, 1, "shuffled", False), (5, 3, 2, "reversed", True), (8, 1, 4, "same", False),
    (8, 1, 1, "reversed", True), (33, 1, 1, "shuffled", False), (40, 2, 4, "reversed", False), (40, 1, 1, "same", True)]]


def test_near_coincident_stacks(gpu):
    rng = np.random.default_rng(2)
    seen, kept_not_least = set(), 0
    decided_not_least = 0
    for K, ulps, per_leaf, order, oblique in STACKS:
        fs, rot = stack_scene(rng, K, ulps, per_leaf, order, oblique)
        o, d = stack_rays(rng, rot)
        what = f"stack K={K} ulps={ulps} per_leaf={per_leaf} {order} oblique={oblique}"
        res = run(gpu, fs, {"stack": (o, d)}, what, SMALL_TREE)
        seen |= outcomes(res, "stack")
        if K <= 8:
            nl = least_t_differs(fs, o, d)
            kept_not_least += int(nl.sum())
            p = np.stack([res[k]["stack"] for k in SPLIT_SETTINGS])
            decided_not_least += int((nl & (((p & 0xff) == SPLIT) & ((p >> 8) == DECIDED)).any(0)).sum())
    # the family holds rays whose reference answer is not the triangle with the least t, and the frontier decided some of them
    # (on a B200: 8 such rays, 2 decided by the frontier; the others run along the normal with zero x / y components: sigma = 0)
    assert kept_not_least > 0 and decided_not_least > 0, (kept_not_least, decided_not_least)
    assert {DECIDED, CAND_FULL}.issubset(seen), seen


def test_duplicates_leaf_pair_fan_and_forest(gpu):
    rng = np.random.default_rng(3)
    fs, fam = duplicates(rng)
    run(gpu, fs, fam, "duplicates", SMALL_TREE)
    f, _, _ = O.OracleScene(fs).closest_many(*fam["duplicates"], 1e30)
    assert f.mean() > 0.5
    fs, fam, n_kind = leaf_pair(rng)
    assert n_kind > 0
    res = run(gpu, fs, fam, "leaf pair", SMALL_TREE)
    assert DECIDED in outcomes(res, "leaf pair")
    fs, fam = fan(rng)
    res = run(gpu, fs, fam, "fan", SMALL_TREE)
    assert MANY in outcomes(res, "fan vertex"), outcomes(res, "fan vertex")
    fs, fam = decoy_forest(rng)
    res = run(gpu, fs, fam, "decoy forest", SMALL_TREE, {k: (v, 0) for k, v in SPLIT_SETTINGS.items()})
    assert outcomes(res, "axis") == {STACK_FULL}, outcomes(res, "axis")


def test_sigma_at_its_limits(gpu):
    rng = np.random.default_rng(4)
    fs, _ = stack_scene(rng, 5, 1, 1, "reversed", scale=4.0)
    fam = limit_rays(fs, rng)
    res = run(gpu, fs, fam, "limits", SMALL_TREE)
    fs2, fam2 = lower_m_family(rng)
    res2 = run(gpu, fs2, fam2, "M low", SMALL_TREE)
    fs3, fam3 = late_family(rng)
    assert len(fam3["late"][0]) > 0
    res3 = run(gpu, fs3, fam3, "late", SMALL_TREE)
    # t >= FINF: the same big stack, directions 2^-30 (|a| of IntersectTriangle stays above 1e-4 on squares of side 2^11)
    fs4, rot = stack_scene(rng, 4, 1, 1, "reversed", scale=2.0 ** 10)
    o, d = stack_rays(rng, rot, scale=2.0 ** 10)
    res4 = run(gpu, fs4, {"finf": (o, d * 2.0 ** -30)}, "finf", SMALL_TREE)
    rf, _, rt = O.OracleScene(fs4).closest_many(o, d * 2.0 ** -30, 1e30)
    assert (rf == 1).any() and (rt[rf == 1] == np.float32(FINF)).all()
    for r, f in ((res, fam), (res2, fam2)):
        for name in f:
            got = outcomes(r, name)
            if name.endswith(" out"):
                assert got == {NO_SIGMA}, (name, got)
            else:
                assert NO_SIGMA not in got and DECIDED in got, (name, got)
    assert LATE in outcomes(res3, "late"), outcomes(res3, "late")
    assert T_FINF in outcomes(res4, "finf"), outcomes(res4, "finf")


def test_trees_the_split_may_not_use(gpu):
    rng = np.random.default_rng(6)
    fs = soup(rng)
    rev = reverse_leaf_order(fs)
    fam = {"surface": outside_rays(rev, rng, 400)}
    res = run(gpu, rev, fam, "soup reversed", parked=LONG)    # parked rays go to k_primary_long whatever primary_split says
    for k in SPLIT_SETTINGS:
        assert ((res[k]["surface"] & 0xff) == LONG).any(), k
    fs, rot = stack_scene(rng, 8, 1, 1, "shuffled")
    fs = flat_tree(balanced([[i] for i in range(fs.n_tri)]), fs.tri, rng, reflection=0.0, cam_pos=(0.0, 0.0, 0.0), nest=False)
    o, d = stack_rays(rng, rot)
    res = run(gpu, fs, {"stack": (o, d)}, "not nested", SMALL_TREE)
    got = outcomes(res, "stack")                                # (a ray outside the analysis as well reports sigma = 0)
    assert NOT_NESTED in got and got <= {NO_SIGMA, NOT_NESTED}, got
