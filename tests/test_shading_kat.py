"""The shading arithmetic case by case, at its edges (ct_gpu_debug_shading: shade_color, blend_color, pow_int and the specular
accumulation, the very functions k_shade / k_resolve call) against the oracle's colour helpers and glibc's pow, and end to end
(frames and shade_rays colours) on small scenes whose materials and lights sit at those edges.

The checkers are tests/shade_oracle.c's loops over the pinned oracle (ct_oracle_shade_color, ct_oracle_blend) and glibc's pow;
on the CPU the oracle's float -> uint8_t form is pinned to a direct assignment, and glibc's pow to the correctly rounded x^n."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import cobbletrace_b200 as ct
from cobbletrace_b200 import host
from cobbletrace_b200.sceneio import FlatScene, LT_AMBIENT, LT_POINT, LT_DIRECTIONAL
from oracle import ct_oracle_py as O
from test_shade_rays import canvas_rays, options, oracle_colors, oracle_lib
from test_walk_limits import gpu  # noqa: F401 (fixture)

INT_MIN, INT_MAX = -(1 << 31), (1 << 31) - 1
vp = C.c_void_p
_bound = []


def lib():
    L = oracle_lib()
    if not _bound:
        L.ct_oracle_shade_many.argtypes = [C.c_uint64, vp, vp, vp]
        L.ct_oracle_blend_many.argtypes = [C.c_uint64, vp, vp, vp, vp]
        L.ct_oracle_pow_many.argtypes = [C.c_uint64, vp, vp, vp, vp, vp, vp]
        L.ct_oracle_u8_forms.argtypes = [C.c_uint64, vp, vp, vp]
        for f in (L.ct_oracle_shade_many, L.ct_oracle_blend_many, L.ct_oracle_pow_many, L.ct_oracle_u8_forms):
            f.restype = None
        _bound.append(True)
    return L


def _p(a):
    return None if a is None else a.ctypes.data


def o_shade(color, intensity):
    color, intensity = np.ascontiguousarray(color, np.uint32), np.ascontiguousarray(intensity, np.float32)
    out = np.zeros(color.size, np.uint32)
    lib().ct_oracle_shade_many(color.size, _p(color), _p(intensity), _p(out))
    return out


def o_blend(lc, rc, refl):
    lc, rc, refl = (np.ascontiguousarray(a, t) for a, t in ((lc, np.uint32), (rc, np.uint32), (refl, np.float32)))
    out = np.zeros(lc.size, np.uint32)
    lib().ct_oracle_blend_many(lc.size, _p(lc), _p(rc), _p(refl), _p(out))
    return out


def o_pow(x, e, acc=None, li=None):
    x, e = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(e, np.int32)
    acc = None if acc is None else np.ascontiguousarray(acc, np.float32)
    li = None if li is None else np.ascontiguousarray(li, np.float32)
    pw = np.zeros(x.size, np.float64)
    out = None if acc is None else np.zeros(x.size, np.float32)
    lib().ct_oracle_pow_many(x.size, _p(x), _p(e), _p(acc), _p(li), _p(pw), _p(out))
    return pw, out


def f32(bits):
    return np.atleast_1d(np.asarray(bits, np.int64)).astype(np.uint32).view(np.float32)


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def around(v, k=4):
    """The float v and the k floats on either side of it (bit steps; v > 0)."""
    b = int(bits(np.float32(v)).item())
    return f32(np.arange(b - k, b + k + 1))


def first_bad(got, want, what, inputs):
    bad = np.flatnonzero(got.view(np.uint32 if got.itemsize == 4 else np.uint64) != want.view(np.uint32 if want.itemsize == 4 else np.uint64))
    if bad.size:
        i = bad[0]
        pytest.fail(f"{what}: {bad.size} of {got.size} cases differ; first {i}: " +
                    ", ".join(f"{k} = {v[i]!r}" for k, v in inputs.items()) + f": device {got[i]!r} against {want[i]!r}")


# ---- case sets -------------------------------------------------------------------------------------------------------------------
INTENSITIES = np.array([0.0, -0.0, f32(1)[0], 0.5, f32(0x3f7fffff)[0], 1.0, f32(0x3f800001)[0], 2.0, -1.0, -1e10, 1e10, np.inf, -np.inf,
                        np.nan], np.float32)


def sampled_intensities(rng, n):
    """Raw float bit patterns; k/255 +- a few ulps for k = 0..256 (where v * 255 crosses an integer); |v * 255| near 2^31."""
    raw = f32(rng.integers(0, 1 << 32, n // 3))
    steps = np.concatenate([around(np.float32(k) / np.float32(255), 6) for k in range(1, 257)] + [f32(np.arange(0, 8))])
    edge = np.concatenate([around(np.float32(2.0 ** 31 / 255), 64), around(np.float32(2.0 ** 31), 8), around(np.float32(2.0 ** 32 / 255), 16)])
    edge = np.concatenate([edge, -edge, -steps])
    near = np.concatenate([steps, edge])
    return np.concatenate([raw, near[rng.integers(0, near.size, n - raw.size)]])


def reflections():
    r = [0.0, -0.0, f32(1)[0], 2.0 ** -24, 0.5, f32(0x3f7fffff)[0], f32(0x3f800001)[0], 2.0, 255.0, 1e7, 1e10, np.finfo(np.float32).max,
         np.inf, -np.inf, np.nan, -1.0, -1e7]
    return np.concatenate([np.array(r, np.float32), around(np.float32(2.0 ** 31 / 255), 4), around(np.float32(2.0 ** 31 / 254), 2),
                           around(np.float32(2.0 ** 31 / 128), 2), around(np.float32(2.0 ** 31), 2)])


def pow_xs(rng, n_random=2000):
    """Floats in (0, 1 + 2^-20] (qv may round above 1): 1 and the 64 floats below it, the 8 above up to 1 + 2^-20, random bit
    patterns, the bottom of the range; and 0 and NaN, which pow_int leaves to pow()."""
    one = int(bits(np.float32(1.0)).item())
    near1 = f32(np.arange(one - 64, one + 9))
    raw = f32(rng.integers(1, one, n_random))
    fixed = np.array([f32(1)[0], 2.0 ** -126, 1e-30, 1e-10, 1e-3, 0.1, 0.25, 0.5, 0.9, 0.99, 0.999999, 0.0, np.nan], np.float32)
    return np.concatenate([near1, raw, fixed])


def pow_es():
    e = [0, 1, 2, 3, 10, 500, INT_MAX, -2, -3, -10, -500, -(1 << 20), INT_MIN, (1 << 20) + 1, 1 << 20]
    for k in range(1, 32):
        e += [(1 << k) - 1, (1 << k) + 1] if (1 << k) + 1 <= INT_MAX else [(1 << k) - 1]
    return np.array(sorted(set(e)), np.int64).astype(np.int32)


def log_uniform_ints(rng, n):
    """Ints of either sign whose magnitudes are spread evenly over 0 .. 31 octaves (most x^n of uniform ints leave the double range)."""
    m = np.floor(2.0 ** (rng.random(n) * 31)).astype(np.int64)
    return np.where(rng.random(n) < 0.5, -m, m).astype(np.int32)


def pow_cases(rng):
    """The grid of pow_xs x pow_es, then 10^6 random ints (half uniform, half log-uniform) with random x of the same set."""
    xs, es = pow_xs(rng), pow_es()
    X, E = np.meshgrid(xs, es, indexing="ij")
    rx = xs[rng.integers(0, xs.size, 1_000_000)]
    re = np.concatenate([rng.integers(INT_MIN, INT_MAX, 500_000, endpoint=True).astype(np.int32), log_uniform_ints(rng, 500_000)])
    return np.concatenate([X.ravel(), rx]), np.concatenate([E.ravel(), re])


def accumulators(rng, x, e):
    """(I, li) per case: a third random, a third with li * pow(x, e) about half an ulp of I (the sum next to a float midpoint), a
    third I = 0 with li of either sign."""
    n = x.size
    pw, _ = o_pow(x, e)
    k = rng.integers(0, 3, n)
    acc = (rng.random(n) * 2).astype(np.float32)
    li = (rng.random(n) * 1.5 - 0.25).astype(np.float32)
    ulp = np.spacing(acc).astype(np.float64)
    with np.errstate(all="ignore"):
        mid = (ulp / 2 / pw).astype(np.float32)
    take = (k == 1) & np.isfinite(mid) & (mid != 0)
    li[take] = mid[take]
    acc[k == 2] = 0.0
    return acc, li


# ---- CPU: the checkers themselves -----------------------------------------------------------------------------------------------
def test_oracle_conversion_is_the_direct_assignment():
    """(uint8_t)(int)c -- the oracle's form -- equals a double -> uint8_t assignment compiled with the oracle's flags, across
    +-2^31, +-2^32, inf and NaN; and ct_oracle_blend's channels are that conversion of wl * l + wr * r (so a reflection of 1e7
    blends 0x00 where 2^31 is passed, not a saturated 0xff)."""
    vals = [0.0, -0.0, 0.5, 255.0, 255.9, 256.0, -1.0, -255.5, np.inf, -np.inf, np.nan, 1e300, -1e300]
    for base in (2.0 ** 31, 2.0 ** 32, 2.0 ** 31 - 1, 2.0 ** 31 + 1, 2.0 ** 33):
        for s in (1.0, -1.0):
            b = s * base
            vals += [b, b - 0.5, b + 0.5, b - 1, b + 1, np.nextafter(b, 0), np.nextafter(b, np.inf), np.nextafter(b, -np.inf)]
    rng = np.random.default_rng(1)
    c = np.concatenate([np.array(vals), rng.uniform(-2.0 ** 34, 2.0 ** 34, 100_000), rng.uniform(-600, 600, 100_000)])
    via, direct = np.zeros(c.size, np.uint8), np.zeros(c.size, np.uint8)
    lib().ct_oracle_u8_forms(c.size, _p(c), _p(via), _p(direct))
    assert np.array_equal(via, direct), c[np.flatnonzero(via != direct)[:8]]
    assert via[c.size - 200_000 + np.argmax(c[-200_000:] >= 2.0 ** 31)] == 0          # cvttsd2si: 0x80000000
    # the oracle's blend against the conversion, channel by channel
    refl = np.concatenate([reflections(), f32(rng.integers(0, 1 << 32, 20_000))])
    l, r = rng.integers(0, 256, refl.size), rng.integers(0, 256, refl.size)
    with np.errstate(all="ignore"):
        wl = (np.float32(1) - refl).astype(np.float64)
        cc = wl * l + refl.astype(np.float64) * r
    via, direct = np.zeros(cc.size, np.uint8), np.zeros(cc.size, np.uint8)
    lib().ct_oracle_u8_forms(cc.size, _p(cc), _p(via), _p(direct))
    got = o_blend(l, r, refl) & 0xff
    assert np.array_equal(got, direct)
    assert o_blend([0], [0xffffff], [1e7])[0] == 0 and o_blend([0], [0xffffff], [0.5])[0] == 0x7f7f7f


def ulps_from_double(mpmath, x, n):
    """(the correctly rounded x^n, (x^n - that double) in its ulps) with 200-bit mpmath."""
    with mpmath.workprec(200):
        v = mpmath.mpf(float(x)) ** int(n)
        d = float(v)                                           # mpf -> float rounds to nearest, ties to even
        return d, float((v - mpmath.mpf(d)) / mpmath.mpf(np.spacing(abs(d))))


def test_glibc_pow_is_correctly_rounded_but_at_halfway_cases():
    """glibc's pow(x, n) against the correctly rounded x^n (mpmath) on the pow case set, wherever x^n is a normal double.  They
    differ only where x^n lies within 0.02 ulp of a rounding midpoint (glibc's bound is 0.52 ulp), exact midpoints among them
    (x^3 of a float with 18 significant bits), which glibc does not always round to even.  So "the device is correctly rounded" and
    "the device equals glibc" are the same claim everywhere else, and test_pow checks both."""
    mpmath = pytest.importorskip("mpmath")
    rng = np.random.default_rng(2)
    xs, es = pow_xs(rng), pow_es()
    X, E = np.meshgrid(xs, es, indexing="ij")
    x = np.concatenate([X.ravel(), xs[rng.integers(0, xs.size, 200_000)]])
    e = np.concatenate([E.ravel(), rng.integers(INT_MIN, INT_MAX, 100_000, endpoint=True).astype(np.int32), log_uniform_ints(rng, 100_000)])
    ok = np.isfinite(x) & (x > 0)
    x, e = x[ok], e[ok]
    pw, _ = o_pow(x, e)
    normal = np.isfinite(pw) & (np.abs(pw) >= np.finfo(np.float64).tiny)
    assert int(normal.sum()) > 40_000
    bad = []
    for xi, ei, p in zip(x[normal].tolist(), e[normal].tolist(), pw[normal].tolist()):
        cr, off = ulps_from_double(mpmath, xi, ei)
        if cr != p:
            bad.append((xi, ei, off))
            assert abs(abs(off) - 0.5) < 0.02 and abs(p - cr) == np.spacing(abs(cr)), (xi, ei, p, cr, off)
    assert len(bad) < 100, bad[:10]
    print(f"glibc pow: {len(bad)} of {int(normal.sum())} results not correctly rounded, "
          f"{sum(abs(abs(o) - 0.5) == 0 for _, _, o in bad)} of them at exact midpoints")


# ---- GPU: the primitives, bit for bit ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_colors_exhaustive(gpu):
    """Every 24-bit colour at 14 intensities: 0, -0, the smallest subnormal, 0.5, 1 and its neighbours, 2, -1, +-1e10, +-inf, NaN."""
    color = np.arange(1 << 24, dtype=np.uint32)
    for v in INTENSITIES:
        inten = np.full(color.size, v, np.float32)
        got = gpu.debug_shading(color=color, intensity=inten)["shaded"]
        first_bad(got, o_shade(color, inten), f"shade_color at intensity {v!r}", dict(color=color))


@pytest.mark.gpu
def test_colors_sampled(gpu):
    rng = np.random.default_rng(3)
    n = 10_000_000
    color = rng.integers(0, 1 << 24, n).astype(np.uint32)
    inten = sampled_intensities(rng, n)
    got = gpu.debug_shading(color=color, intensity=inten)["shaded"]
    first_bad(got, o_shade(color, inten), "shade_color", dict(color=color, intensity=inten))


@pytest.mark.gpu
def test_blend(gpu):
    """All 256 x 256 channel pairs (in each channel) at the edge reflections, then 10^6 reflections drawn as raw float bits.  A
    channel that reaches 2^31 (reflection >= 2^31 / 255 with the reflected channel above the local one) is 0x00, as x86 truncates."""
    l, r = (a.ravel().astype(np.uint32) for a in np.meshgrid(np.arange(256), np.arange(256), indexing="ij"))
    lc, rc = l | ((255 - l) << 8) | (r << 16), r | ((255 - r) << 8) | (l << 16)
    for refl in reflections():
        rf = np.full(lc.size, refl, np.float32)
        got = gpu.debug_shading(lc=lc, rc=rc, reflection=rf)["blended"]
        first_bad(got, o_blend(lc, rc, rf), f"blend_color at reflection {refl!r}", dict(lc=lc, rc=rc))
    rng = np.random.default_rng(4)
    n = 1_000_000
    lc, rc = (rng.integers(0, 1 << 24, n).astype(np.uint32) for _ in range(2))
    rf = f32(rng.integers(0, 1 << 32, n))
    got = gpu.debug_shading(lc=lc, rc=rc, reflection=rf)["blended"]
    first_bad(got, o_blend(lc, rc, rf), "blend_color", dict(lc=lc, rc=rc, reflection=rf))


@pytest.mark.gpu
def test_pow_and_the_specular_accumulation(gpu):
    """pow_int's double is the correctly rounded x^n wherever |x^n| is in [2^-900, 2^900]: glibc's, except at the halfway cases
    glibc does not round to even; the float accumulation equals glibc's everywhere."""
    rng = np.random.default_rng(5)
    x, e = pow_cases(rng)
    acc, li = accumulators(rng, x, e)
    want_pw, want_acc = o_pow(x, e, acc, li)
    out = gpu.debug_shading(x=x, e=e, acc=acc, li=li)
    inside = (np.abs(want_pw) >= 2.0 ** -900) & (np.abs(want_pw) <= 2.0 ** 900)
    assert int(inside.sum()) > 100_000
    # where glibc is not correctly rounded (x^n within 0.02 ulp of a midpoint, see the CPU test above) the device must be
    differ = np.flatnonzero(inside & (out["pow"].view(np.uint64) != want_pw.view(np.uint64)))
    mpmath = pytest.importorskip("mpmath")
    for i in differ[:1000]:
        cr, off = ulps_from_double(mpmath, x[i], e[i])
        assert out["pow"][i] == cr and abs(abs(off) - 0.5) < 0.02, (
            f"pow_int({x[i]!r}, {e[i]}) = {out['pow'][i]!r}, glibc {want_pw[i]!r}, correctly rounded {cr!r} ({off:+.6f} ulp)")
    assert differ.size < 1000
    print(f"pow_int: {differ.size} of {int(inside.sum())} results differ from glibc's, all where glibc is not correctly rounded")
    first_bad(out["acc"], want_acc, "specular accumulation", dict(x=x, e=e, acc=acc, li=li))


# ---- GPU: end to end ---------------------------------------------------------------------------------------------------------------
SPECULARS = np.array([-1, 0, 1, 2, 3, 10, 500, -2, -7, -500, INT_MIN, INT_MAX, (1 << 20) + 1, 1 << 25], np.int32)
COLORS = np.array([0x000000, 0xffffff, 0x808080, 0x010101, 0x0000ff, 0x00ff00, 0xff0000, 0xff00ff, 0x00ffff, 0xffff00, 0xff0001,
                   0xfe00ff, 0xff01ff, 0x7f00ff, 0x123456, 0xfffffe], np.uint32)


def edge_soup(rng, n_tri, lights):
    """A soup in front of the camera whose materials cross the edge speculars, reflections and colours, with `lights`
    (type, intensity, pos, dir arrays)."""
    c = rng.normal(size=(n_tri, 3)) * 1.5 + np.array([0.0, 0.0, 6.0])
    a, b = rng.normal(size=(n_tri, 3)) * 0.8, rng.normal(size=(n_tri, 3)) * 0.8
    tri = np.concatenate([c - (a + b) / 3, c - (a + b) / 3 + a, c - (a + b) / 3 + b], 1)
    refl = reflections()
    refl = np.concatenate([refl, np.zeros(refl.size, np.float32)])          # half of the triangles do not reflect
    lt, li, lp, ld = lights
    fs = FlatScene(tri=tri, mat_color=COLORS[rng.integers(0, COLORS.size, n_tri)], mat_specular=SPECULARS[rng.integers(0, SPECULARS.size, n_tri)],
                   mat_reflection=refl[rng.integers(0, refl.size, n_tri)], light_type=lt, light_intensity=li, light_pos=lp, light_dir=ld,
                   cam_pos=np.zeros(3), cam_rot=np.eye(3).reshape(9))
    return host.HostScene.from_flat(fs).to_flat(with_bvh=True)


def light_set(rng, n, ambient_at=(31, 32, 63, 64), intensities=None):
    lt = np.where(rng.random(n) < 0.5, LT_POINT, LT_DIRECTIONAL).astype(np.int32)
    lt[[i for i in ambient_at if i < n]] = LT_AMBIENT
    li = (rng.random(n) * 0.04 + 0.005).astype(np.float32) if intensities is None else np.asarray(intensities, np.float32)
    lp = rng.normal(size=(n, 3)) * 4 + np.array([0.0, 0.0, 3.0])
    ld = rng.normal(size=(n, 3))
    ld[:, 2] = -np.abs(ld[:, 2])
    return lt, li, lp, ld


def shading_point(fs, o, d):
    """The shading point of the ray (o, d), as TraceRay computes it (raythread.cpp:360: org + double(t) * dir, no FMA)."""
    found, _, t = O.OracleScene(fs).closest(o, d)
    assert found
    return np.asarray(o) + np.float64(np.float32(t)) * np.asarray(d)


def edge_scenes():
    rng = np.random.default_rng(6)
    out = {}
    for n in (31, 32, 33, 64, 65, 97):
        out[f"lights{n}"] = edge_soup(rng, 160, light_set(rng, n))
    # a point light on a shading point (a zero light ray), a zero directional vector, next to ordinary lights
    fs = edge_soup(rng, 160, light_set(rng, 4, ambient_at=(0,), intensities=[0.2, 0.5, 0.4, 0.3]))
    o, d = np.zeros(3), np.array([0.02, -0.01, 1.0])
    lp, ld = fs.light_pos.copy(), fs.light_dir.copy()
    lt = fs.light_type.copy()
    lt[1], lt[2] = LT_POINT, LT_DIRECTIONAL
    lp[1], ld[2] = shading_point(fs, o, d), 0.0
    out["zero_rays"] = dataclasses.replace(fs, light_type=lt, light_pos=lp, light_dir=ld)
    # non-finite, negative and huge intensities, on ambient, point and directional lights
    for name, vals in (("nan", [np.nan, 0.3]), ("negative", [-0.7, -1e10]), ("huge", [1e30, 3.0]), ("inf", [np.inf, -np.inf])):
        lts = light_set(rng, 6, ambient_at=(5,))
        li = np.array([0.2, vals[0], 0.3, vals[1], 0.1, 0.1], np.float32)
        out[f"intensity_{name}"] = edge_soup(rng, 160, (lts[0], li, lts[2], lts[3]))
        li2 = li.copy()
        li2[5] = vals[0]                                                     # ... on the ambient light too
        out[f"ambient_{name}"] = edge_soup(rng, 120, (lts[0], li2, lts[2], lts[3]))
    return out


@pytest.fixture(scope="module")
def scenes():
    return edge_scenes()


@pytest.mark.gpu
@pytest.mark.parametrize("reuse", [1, 0])
@pytest.mark.parametrize("depth", [0, 1, 2, 15])
def test_edge_scenes_end_to_end(depth, reuse, scenes, gpu):
    """Frames (render_tile) and shade_rays colours on scenes whose materials and lights sit at the edges, against the oracle's frame
    and ct_oracle_trace_many, at depths 0 / 1 / 2 / 15, with and without shadow-ray reuse."""
    import torch
    W = H = 48
    rng = np.random.default_rng(depth * 2 + reuse)
    for name, fs in scenes.items():
        oframe, _, _ = O.OracleScene(fs).render(W, H, max_depth=depth, want_hits=False)
        y, x = np.mgrid[-H // 2:H // 2, -W // 2:W // 2]
        o, d = canvas_rays(fs, H, x.ravel() + rng.random(x.size) - 0.5, y.ravel() + rng.random(x.size) - 0.5)
        if name == "zero_rays":
            o, d = np.vstack([o, np.zeros(3)]), np.vstack([d, [0.02, -0.01, 1.0]])
        want = oracle_colors(fs, o, d, depth)
        with options(shadow_reuse=reuse):
            gpu.upload(fs, W, H, max_depth=depth)
            gpu.render_tile()
            frame = gpu.readback()
            got = gpu.shade_rays(torch.from_numpy(np.ascontiguousarray(o)).to("cuda:0"), torch.from_numpy(np.ascontiguousarray(d)).to("cuda:0"))
            got = got.cpu().numpy().view(np.uint32)
        assert np.array_equal(frame, oframe), f"{name} depth {depth} reuse {reuse}: {int((frame != oframe).sum())} pixels differ"
        first_bad(got, want, f"{name} depth {depth} reuse {reuse}: shade_rays", dict(o=o, d=d))
