"""The closest-hit walk as an order-free search, checked on the CPU before the kernel (k_primary_split) relies on it.
oracle/ct_oracle.c holds a prototype: any visit order, boxes pruned with a margin against the best t so far, the candidates
within a rounding slop of the minimum replayed in leaf order with the reference's update rules -- or "undecided", where the
caller falls back to the ordered walk.  Every ray the prototype decides must equal the reference-order walk bit for bit
(found, triangle index, tclosest), for both visit orders."""
import numpy as np
import pytest

from oracle import ct_oracle_py as O
from conftest import load_fuzz_case
from test_prehit_prototype import camera_rays


@pytest.mark.parametrize("name,H", [("scene_file_cube", 96), ("scene_import", 96), ("scene_import_bunny", 128), ("pc_big", 96)])
def test_free_walk_equals_reference_walk_on_bundled_scenes(name, H, scene_loader):
    fs = scene_loader(name)
    sc = O.OracleScene(fs)
    rng = np.random.default_rng(7)
    for order in (0, 1):
        for jitter in (0.0, 0.003):
            org, d = camera_rays(fs, H, H, rng, jitter)
            bad, st = O.free_check(sc, org, d, order)
            assert bad == 0, (name, order, jitter, bad, st)
            # the axis-aligned scenes are where a triangle's t and its leaf box's entry distance tie: still decided
            assert st["fallback"] <= 0.02 * st["rays"] + 2 * H, (name, order, jitter, st)    # (x = 0 / y = 0 lines: zero direction component)
        c = fs.tri.reshape(-1, 3).mean(0)
        ext = np.ptp(fs.tri.reshape(-1, 3), axis=0).max()
        org = c + rng.normal(size=(4000, 3)) * ext * 0.7
        bad, st = O.free_check(sc, org, rng.normal(size=(4000, 3)), order)
        assert bad == 0, (name, order, "random", bad, st)


def test_free_walk_equals_reference_walk_on_generated_scenes(golden):
    rng = np.random.default_rng(8)
    for k in golden["fuzz"]:
        fs, _ = load_fuzz_case(k)
        org, d = camera_rays(fs, 48, 48, rng, 0.002)
        for order in (0, 1):
            bad, st = O.free_check(O.OracleScene(fs), org, d, order)
            assert bad == 0, (k, order, bad, st)


@pytest.mark.parametrize("name,H", [("scene_file_cube", 96), ("scene_import", 96), ("scene_import_bunny", 128), ("pc_big", 96)])
def test_frontier_walk_equals_reference_walk(name, H, scene_loader):
    """The same search as a FRONTIER -- up to 32 pending nodes per round, the minimum of t exchanged once per round: what one
    warp finishing one long walk together would do (DESIGN.md 8).  Every decided ray equals the reference-order walk; the rounds a
    walk needs are bounded by the tree's depth, not by the number of boxes the ray grazes."""
    fs = scene_loader(name)
    sc = O.OracleScene(fs)
    rng = np.random.default_rng(9)
    org, d = camera_rays(fs, H, H, rng, 0.002)
    st = O.rounds_check(sc, org, d, 0)
    assert st["differ"] == 0 and st["rays"] == org.shape[0], (name, st)
    assert st["undecided"] <= 0.02 * st["rays"], (name, st)
    c = fs.tri.reshape(-1, 3).mean(0)
    ext = np.ptp(fs.tri.reshape(-1, 3), axis=0).max()
    org = c + rng.normal(size=(3000, 3)) * ext * 0.7
    st = O.rounds_check(sc, org, rng.normal(size=(3000, 3)), 0)
    assert st["differ"] == 0, (name, "random", st)


def test_slop_bound_holds_on_adversarial_cases():
    """sigma = 2^-15 M bounds how much EARLIER than its own box a triangle can seem to be hit (tray_nearest_setup's analysis: < 340 * 2^-24 M).
    Rays aimed at points on and just around triangles -- interiors, edges, vertices; fat, needle and axis-aligned triangles; grazing and
    near-axis directions; near and far origins -- in the reference's arithmetic: the worst observed ratio must stay below the bound."""
    rng = np.random.default_rng(11)
    n = 400_000
    scale = 10.0 ** rng.uniform(-0.5, 1, size=(n, 1))
    p1 = rng.normal(size=(n, 3)) * scale
    e1 = rng.normal(size=(n, 3)) * scale * 10.0 ** rng.uniform(-1.5, 0, size=(n, 1))     # needles included: the two edges' lengths are independent
    e2 = rng.normal(size=(n, 3)) * scale * 10.0 ** rng.uniform(-1.5, 0, size=(n, 1))
    flat = rng.integers(0, 4, size=n)                                   # a quarter each: generic, and flat in x / y / z (zero-thickness boxes)
    for a in range(3):
        e1[flat == a + 1, a] = 0.0; e2[flat == a + 1, a] = 0.0
    tri = np.concatenate([p1, p1 + e1, p1 + e2], axis=1)
    kind = rng.integers(0, 4, size=n)                                   # target: interior, an edge, a vertex, just outside an edge
    u = rng.uniform(0, 1, size=n); v = rng.uniform(0, 1, size=n) * (1 - u)
    u = np.where(kind == 1, rng.uniform(0, 1, size=n), u); v = np.where(kind == 1, 0.0, v)
    u = np.where(kind == 2, rng.integers(0, 2, size=n).astype(float), u); v = np.where(kind == 2, 0.0, v)
    v = np.where(kind == 3, -1e-7 * rng.uniform(0, 1, size=n), v)
    target = p1 + u[:, None] * e1 + v[:, None] * e2
    d = rng.normal(size=(n, 3))
    graze = rng.integers(0, 3, size=n) == 0                             # a third of the rays nearly parallel to an axis plane
    ax = rng.integers(0, 3, size=n)
    d[graze, ax[graze]] *= 10.0 ** rng.uniform(-6, -2, size=int(graze.sum()))
    dist = 10.0 ** rng.uniform(-3, 2, size=(n, 1))
    org = target - d * dist
    passes, worst, skipped = O.slop_check(org, d, tri)
    assert passes > 0.25 * n and skipped < 0.2 * n, (passes, skipped)     # (the misses: just outside an edge, |a| < 1e-4 (bvh.cpp:152), rounding at edges and vertices)
    assert worst <= 340 * 2.0 ** -24, (worst / 2.0 ** -24, "x 2^-24")          # the analysis' bound; sigma = 512 x 2^-24 on top
