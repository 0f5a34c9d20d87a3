"""ct_gpu_build_bvh: the reference's BuildBVH (bvh.cpp:16-120) built on the device, level by level.

CPU: `level_build` restates in numpy the schedule the kernels in ct_bvh_build.cuh run -- one prefix sum of the partition
predicate over all positions per level, the closed-form destinations of the in-place partition, ordered (last operand wins on
ties) reductions for the children's bounds, and the numbering from the tree's shape -- and is checked against the oracle's
BuildBVH on the golden scenes and on adversarial families.

GPU: the device build must give the reference's tree exactly -- every node field, _pad included, and tri_index -- on the golden
scenes (golden.json's bvh_sha256), the fuzz scenes' stored reference trees, the dragon stand-in (host build), and the same
adversarial families at strides 72, 96 and 120."""
import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import api, host, procedural
from oracle import ct_oracle_py as O

from conftest import load_fuzz_case

FIELDS = ("node_min", "node_max", "node_left", "node_first", "node_count", "tri_index")
GOLDEN_SCENES = ["pc_big", "scene_file_cube", "scene_import", "scene_import_bunny"]
F32 = np.float32


# ---- the level-synchronous schedule in numpy ------------------------------------------------------------------------------
def last_fold(vals, starts, lengths, init, is_min):
    """The reference's fold `acc = acc < v ? acc : v` (max: `acc > v`) from `init` over each segment of `vals`, in order:
    the LAST element equal to the extreme, or init when no element reaches it.  Associative, so any grouping that combines
    the earlier operand first gives it -- as k_bb_bounds / k_bb_finish do."""
    red = (np.minimum if is_min else np.maximum).reduceat(vals, starts)
    seg = np.repeat(np.arange(len(starts)), lengths)
    pos = np.where(vals == red[seg], np.arange(len(vals)), -1)
    last = np.maximum.reduceat(pos, starts)
    reaches = red <= init if is_min else red >= init
    return np.where(reaches, vals[last], init)


def level_build(tri):
    tri = np.ascontiguousarray(tri, np.float64).reshape(-1, 9)
    n = tri.shape[0]
    third = np.float64(F32(0.3333))
    cen = (third * ((tri[:, 0:3] + tri[:, 3:6]) + tri[:, 6:9])).astype(F32)       # float(centroid), bvh.cpp:112
    rec_idx = np.arange(n, dtype=np.int64)                                        # the permutation moves whole records
    first, count, left = [0], [n], [0]
    mn, mx = [None], [None]

    def bounds(ids):
        """UpdateNodeBounds (bvh.cpp:30-49) of nodes `ids` over the current record order: 3 vertices per position, in order."""
        st = np.array([first[i] for i in ids]); ln = np.array([count[i] for i in ids])
        pos = np.concatenate([np.arange(s, s + c) for s, c in zip(st, ln)])
        v = tri[rec_idx[pos]].reshape(-1, 3, 3)                                   # [position, vertex, axis]
        for i in ids:
            mn[i] = np.zeros(3); mx[i] = np.zeros(3)
        starts = 3 * (np.cumsum(ln) - ln)
        for a in range(3):
            seq = v[:, :, a].reshape(-1)
            lo = last_fold(seq, starts, 3 * ln, np.float64(F32(1e30)), True)
            hi = last_fold(seq, starts, 3 * ln, -np.float64(F32(1e30)), False)
            for j, i in enumerate(ids):
                mn[i][a] = lo[j]; mx[i][a] = hi[j]

    def plan(i):
        ext = mx[i] - mn[i]
        axis = 0
        if ext[1] > ext[0]:
            axis = 1
        if ext[2] > np.float64(F32(ext[axis])):
            axis = 2
        with np.errstate(all="ignore"):
            split = F32(mn[i][axis]) + F32(ext[axis]) * F32(0.5)
        return axis, split

    bounds([0])
    levels = [(0, 1)]
    while True:
        b, e = levels[-1]
        plans = {i: plan(i) for i in range(b, e) if count[i] > 2}
        small = np.zeros(n + 1, np.int64)
        for i, (axis, split) in plans.items():
            r = slice(first[i], first[i] + count[i])
            with np.errstate(invalid="ignore"):
                small[r] = cen[rec_idx[r], axis] < split
        S = np.concatenate([[0], np.cumsum(small[:n])])                            # exclusive prefix sum, S[n] = total
        new_idx = rec_idx.copy()
        splits = []
        for i in plans:
            f, c = first[i], count[i]
            k = S[f + c] - S[f]
            n_pairs = k - (S[f + k] - S[f])
            q = np.arange(c)
            sm = S[f + q] - S[f]
            is_small = small[f + q] == 1
            ll_pos = np.zeros(max(n_pairs, 1), np.int64); before = np.zeros(max(n_pairs, 1), np.int64)
            hi = c - 1
            sel = is_small & (q >= k)
            r_ = k - (sm[sel] + 1)
            w = r_ + 1 < n_pairs
            before[r_[w] + 1] = (r_[w] + 1) + ((c - k) - (q[sel][w] + 1 - (sm[sel][w] + 1)))
            if n_pairs:
                hi = q[sel][r_ == n_pairs - 1][0] - 1
            sel2 = ~is_small & (q < k)
            ll_pos[q[sel2] - sm[sel2]] = q[sel2]
            dest = np.empty(c, np.int64)
            a = is_small & (q < k); dest[a] = q[a]
            a = is_small & (q >= k); dest[a] = ll_pos[k - (sm[a] + 1)]
            a = ~is_small & (q < k); dest[a] = c - 1 - before[q[a] - sm[a]]
            a = ~is_small & (q >= k)
            above = k - sm[a]
            d = np.where(above < n_pairs, c - 1 - (above + 1) - ((c - k) - (q[a] + 1 - sm[a])), np.where(q[a] > k, q[a] - 1, hi))
            dest[a] = d
            assert np.array_equal(np.sort(dest), q)
            new_idx[f + dest] = rec_idx[f + q]
            if k != 0 and k != c:
                splits.append((i, k))
        rec_idx = new_idx
        if not splits:
            break
        for m, (i, k) in enumerate(splits):                                 # children in level order
            l = e + 2 * m
            left[i] = l
            f, c = first[i], count[i]
            first += [f, f + k]; count += [k, c - k]; left += [0, 0]; mn += [None, None]; mx += [None, None]
        levels.append((e, e + 2 * len(splits)))
        bounds(list(range(e, e + 2 * len(splits))))
    # numbering from the shape: interior counts bottom-up, pre-order ranks top-down, left(X) = 1 + 2 rank(X)
    U = levels[-1][1]
    inner = np.zeros(U, np.int64); rank = np.zeros(U, np.int64); fin = np.zeros(U, np.int64)
    for b, e in reversed(levels):
        for i in range(b, e):
            if left[i]:
                inner[i] = 1 + inner[left[i]] + inner[left[i] + 1]
    out = dict(node_min=np.zeros((U, 3)), node_max=np.zeros((U, 3)), node_left=np.zeros(U, np.uint32),
               node_first=np.zeros(U, np.uint32), node_count=np.zeros(U, np.uint32))
    for b, e in levels:
        for i in range(b, e):
            if left[i]:
                l = left[i]
                fin[l] = 1 + 2 * rank[i]; fin[l + 1] = fin[l] + 1
                rank[l] = rank[i] + 1; rank[l + 1] = rank[i] + 1 + inner[l]
            j = fin[i]
            out["node_min"][j], out["node_max"][j] = mn[i], mx[i]
            out["node_left"][j] = fin[left[i]] if left[i] else 0
            out["node_first"][j] = first[i]
            out["node_count"][j] = 0 if left[i] else count[i]
    out["tri_index"] = rec_idx.astype(np.uint32)
    return out, len(levels)


def same_tree(a, b):
    """Every field bit for bit (bounds compared as bit patterns: +0.0 / -0.0 and the 1e30f start values matter)."""
    for k in FIELDS:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.dtype == np.float64:
            x, y = x.view(np.uint64), y.view(np.uint64)
        if x.shape != y.shape or not np.array_equal(x, y):
            return k
    return None


# ---- adversarial families -----------------------------------------------------------------------------------------------
def soup(rng, n, scale=1.0):
    c = rng.uniform(-10, 10, (n, 1, 3)) * scale
    return (c + rng.normal(size=(n, 3, 3)) * 0.3 * scale).reshape(n, 9)


def same_centroid(rng, n=40):
    """Every centroid exactly 0 on every axis and the split plane below it: the root cannot be split, but the partition has
    permuted it (the order inside the leaf is the test order)."""
    a = rng.uniform(1, 2, n); b = rng.uniform(0.1, 0.4, n)
    z = np.zeros(n)
    return np.stack([-a, z, z, a / 2, b, z, a / 2, -b, z], 1)


def on_the_plane(rng):
    """Centroids exactly on the root's split plane in float, some equal in float but not in double, between two triangles
    that fix the root's box."""
    box = [[0.0, 0, 0, 0.0, 1, 0, 0.0, 0, 1], [1.0, 0, 0, 1.0, 1, 0, 1.0, 0, 1]]
    split = F32(0.0) + F32(1.0) * F32(0.5)
    third = np.float64(F32(0.3333))
    out = []
    base = 0.5 / (3 * third)
    for j in range(-40, 41):
        x = base * (1 + j * 2.0 ** -40)
        if F32(third * ((x + x) + x)) in (split, np.nextafter(split, F32(1)), np.nextafter(split, F32(0))):
            out.append([x, 0.4, 0.4, x, 0.6, 0.4, x, 0.4, 0.6])
    assert len(out) > 10
    t = np.array(box + out + box, np.float64)
    return np.concatenate([t, t[::-1] + 0.0])


def signed_zeros():
    """Coordinates +0.0 and -0.0 in every order on every axis (bounds keep the later one on ties)."""
    out = []
    for bits in range(64):
        s = [(-0.0 if bits >> j & 1 else 0.0) for j in range(6)]
        out.append([s[0], s[1], 1.0, 2.0, s[2], s[3], s[4], 3.0, s[5]])
        out.append([s[5], 1.5, s[4], s[3], s[2], 0.5, 1.0, s[1], s[0]])
    return np.array(out)


def beyond_float(rng):
    """Vertices beyond +-1e30 (they never move the initial bounds) and beyond the float range (infinite float extent, NaN split)."""
    t = soup(rng, 60)
    t[::5, 0] = 1e31; t[1::7, 4] = -1e35; t[2::11, 8] = 1e300; t[3::13, 3] = -1e300; t[4::9, 1] = 3e38
    return t


def axis_rounding(rng, n=400):
    """A root box with ext[0] = 1 + 2^-30 and ext[2] = 1 + 2^-31: ext[2] < ext[0] in double, but ext[2] > (double)(float)ext[0] = 1,
    so BuildBVH splits along z (bvh.cpp:63-65)."""
    X, Z = 1 + 2.0 ** -30, 1 + 2.0 ** -31
    box = [[0.0, 0.0, 0.0, X, 0.5, Z, 0.0, 0.5, 0.0]]
    c = np.column_stack([rng.uniform(0.1, 0.9, n), rng.uniform(0.1, 0.4, n), rng.uniform(0.1, 0.9, n)])
    t = np.repeat(c, 3, axis=0).reshape(n, 9) + rng.uniform(-0.05, 0.05, (n, 9))
    return np.concatenate([box, t])


def duplicates(rng, n=100000):
    pool = soup(rng, 50)
    return pool[rng.integers(0, 50, n)]


def geometric(n, ratio=0.45):
    """Centroids in a geometric series along x: BuildBVH peels one triangle off per level, a comb of depth about n, until the
    float centroids run out of range."""
    c = ratio ** np.arange(n)
    s = 0.1 * c
    return np.stack([c - s, -s, -s, c + s, s, -s, c, -s, s], 1)


def tree_depth(t):
    left, count = t["node_left"], t["node_count"]
    best, st = 0, [(0, 1)]
    while st:
        i, d = st.pop()
        best = max(best, d)
        if count[i] == 0:
            st += [(int(left[i]), d + 1), (int(left[i]) + 1, d + 1)]
    return best


def comb_of_depth(depth):
    for n in range(depth - 5, depth + 10):
        t = geometric(n)
        if tree_depth(O.build_bvh(t)) == depth:
            return t
    raise AssertionError(f"no geometric comb of depth {depth}")


# thresholds of the device build: warp (32), CTA (256 threads, 256 positions per chunk of k_bb_bounds), scan tile (1024)
THRESHOLDS = [31, 32, 33, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 2047, 2048, 2049]


def families(rng):
    fam = {f"n={n}": soup(rng, n) for n in (1, 2, 3)}
    fam["same centroid"] = same_centroid(rng)
    fam["identical"] = np.tile(soup(rng, 1), (37, 1))
    fam["on the plane"] = on_the_plane(rng)
    fam["signed zeros"] = signed_zeros()
    fam["beyond float"] = beyond_float(rng)
    fam["axis rounding"] = axis_rounding(rng)
    fam["grid"] = np.round(soup(rng, 3000) * 2) / 2            # many centroids on and next to split planes
    for n in THRESHOLDS:
        fam[f"soup {n}"] = soup(rng, n)
    fam["comb 96"] = comb_of_depth(96)
    fam["comb 97"] = comb_of_depth(97)
    fam["deepest comb"] = geometric(400)
    return fam


def test_families_reach_what_they_are_for():
    assert tree_depth(O.build_bvh(geometric(400))) > 97
    t = O.build_bvh(axis_rounding(np.random.default_rng(1)))
    left = t["node_left"][0]
    assert t["node_min"][left + 1][2] > 0.4 and t["node_min"][left + 1][0] < 0.1  # the root was split along z


# ---- CPU: the schedule against the oracle ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_level_schedule_golden(name, scene_loader):
    fs = scene_loader(name)
    got, _ = level_build(fs.tri)
    assert same_tree(got, {k: getattr(fs, k) for k in FIELDS}) is None


def test_level_schedule_adversarial():
    rng = np.random.default_rng(7)
    fam = families(rng)
    fam["duplicates"] = duplicates(rng)
    for what, t in fam.items():
        got, _ = level_build(t)
        bad = same_tree(got, O.build_bvh(t))
        assert bad is None, f"{what}: {bad} differs"


def test_level_schedule_fuzz():
    for k in range(0, 20, 4):
        fs, _ = load_fuzz_case(f"{k:02d}")
        got, _ = level_build(fs.tri)
        assert same_tree(got, {f: getattr(fs, f) for f in FIELDS}) is None, k


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
def device_build(tri, stride=72, capacity=None):
    """ct_gpu_build_bvh on raw triangles; returns (tree dict, the raw node records)."""
    L = api.load_library()
    tri = np.ascontiguousarray(tri, np.float64).reshape(-1, 9)
    n = tri.shape[0]
    if stride != 72:
        wide = np.full((n, stride // 8), np.nan)
        wide[:, :9] = tri
        tri = wide
    cap = max(2 * n - 1, 1) if capacity is None else capacity
    nodes = np.frombuffer(b"\xab" * (64 * max(cap, 1)), api.NODE_DT).copy()       # every byte the call leaves alone shows
    idx = np.zeros(max(n, 1), np.uint32)
    used = L.ct_gpu_build_bvh(0, n, api._ptr(tri), stride, api._ptr(nodes), cap, api._ptr(idx))
    if used < 0:
        raise ct.CtError(used, L.ct_gpu_last_error().decode())
    nodes = nodes[:used]
    assert not nodes["pad"].any()
    return dict(node_min=nodes["min"], node_max=nodes["max"], node_left=nodes["left"], node_first=nodes["first"],
                node_count=nodes["count"], tri_index=idx[:n]), nodes


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_SCENES)
def test_device_build_golden(name, scene_loader, golden):
    fs = scene_loader(name)
    built = api.build_bvh(fs.without_bvh())
    assert built.bvh_digest() == golden["scenes"][name]["bvh_sha256"]
    tree, _ = device_build(fs.tri)
    assert same_tree(tree, {k: getattr(fs, k) for k in FIELDS}) is None


@pytest.mark.gpu
def test_device_build_fuzz():
    for k in range(20):
        fs, _ = load_fuzz_case(f"{k:02d}")
        tree, _ = device_build(fs.tri, stride=(72, 96, 120)[k % 3])
        bad = same_tree(tree, {f: getattr(fs, f) for f in FIELDS})
        assert bad is None, f"fuzz_{k:02d}: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [72, 96, 120])
def test_device_build_adversarial(stride):
    rng = np.random.default_rng(11)
    fam = families(rng)
    if stride == 72:
        fam["duplicates"] = duplicates(rng)
    for what, t in fam.items():
        tree, _ = device_build(t, stride=stride)
        bad = same_tree(tree, O.build_bvh(t))
        assert bad is None, f"{what} (stride {stride}): {bad} differs"


@pytest.mark.gpu
def test_device_build_dragon_standin(tmp_path):
    scene, n = procedural.write_dragon_standin(str(tmp_path))
    fs = host.HostScene.load(scene, base_dir=str(tmp_path)).to_flat(with_bvh=True)
    tree, _ = device_build(fs.tri)
    assert same_tree(tree, {k: getattr(fs, k) for k in FIELDS}) is None


@pytest.mark.gpu
def test_device_build_errors():
    t = soup(np.random.default_rng(3), 10)
    with pytest.raises(ct.CtError) as e:
        device_build(t, capacity=18)
    assert e.value.code == -1
    with pytest.raises(ct.CtError) as e:
        device_build(np.zeros((0, 9)), capacity=1)
    assert e.value.code == -1
    with pytest.raises(ct.CtError) as e:
        device_build(t, stride=76)
    assert e.value.code == -1
    tree, _ = device_build(t, capacity=19)
    assert same_tree(tree, O.build_bvh(t)) is None


@pytest.mark.gpu
def test_device_build_leaves_a_resident_scene_alone(scene_loader):
    fs = scene_loader("scene_file_cube").with_reflection(0.5)
    r = ct.GpuRenderer(0).upload(fs, 64, 64, max_depth=2)
    try:
        r.render_tile()
        before = r.readback().copy()
        bunny = scene_loader("scene_import_bunny")
        assert api.build_bvh(bunny.without_bvh()).bvh_digest() == bunny.bvh_digest()
        r.render_tile()
        assert np.array_equal(r.readback(), before)
    finally:
        r.shutdown()
