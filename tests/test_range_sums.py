"""The sample-range reduction of k_render (DESIGN.md §5), held bit for bit to an exact sum of its partials.

A path's radiance depends only on (seed, pixel, sample), and a render with sample_count = 1, sample_begin = s and
sample_ranges = 1 writes sample s's float value X[p, s] as it is.  So every partial sum the kernel forms can be rebuilt
outside it: range c of a pixel with m samples covers k in [cum[c]*m/total, cum[c+1]*m/total) (rtnw_plan_sample_ranges),
summed in float32 in sample order from 0.  The expected pixel is then computed in Python integers: every finite partial
rounded once to a multiple of 2^-54 (ties to even), the multiples summed exactly, the sum rounded once to float32 (ties to
even, +-inf beyond FLT_MAX); a NaN partial, or +inf and -inf together, give NaN, +inf or -inf alone give that infinity.
With one range there is nothing to reduce and the pixel is its float partial.

The magnitude wall is a wall of emitting rectangles seen head-on, one constant emission per tile, over the whole float
range (0 to FLT_MAX, the infinities and NaN, and values that are ties at the 2^-54 unit); the tile edges fall inside
pixels, so boundary pixels mix neighbouring emissions."""
import ctypes as C
import math
import random
from fractions import Fraction

import numpy as np
import pytest

from test_sample_ranges import _pixel_sample_count

UNIT_LOG2 = -54  # the reduction's unit: include/rtnw.h, rtnw_plan_sample_ranges
F32_MAX = float(np.finfo(np.float32).max)


# ------------------------------------------------------------------------------------------------ the exact reference
def to_float32_rne(n: int, unit_log2: int) -> np.float32:
    """n * 2^unit_log2 rounded once to float32, to nearest with ties to even, +-inf when it rounds to 2^128 or beyond.
    (float(n) would round to 53 bits first and so round twice.)"""
    if n == 0:
        return np.float32(0.0)
    sign, a = (-1.0 if n < 0 else 1.0), abs(n)
    lsb = max(a.bit_length() - 24 + unit_log2, -149)  # exponent of the last significand bit float32 keeps
    sh = lsb - unit_log2
    if sh > 0:
        q, rem, half = a >> sh, a & ((1 << sh) - 1), 1 << (sh - 1)
        if rem > half or (rem == half and q & 1):
            q += 1
    else:
        q, lsb = a, unit_log2
    if q.bit_length() + lsb > 128:
        return np.float32(sign * math.inf)
    return np.float32(sign * math.ldexp(q, lsb))  # q < 2^25: exact in a double, and representable in float32


def round_to_unit(parts: np.ndarray, unit_log2: int = UNIT_LOG2) -> np.ndarray:
    """finite float32 values -> the nearest multiples of 2^unit_log2 (ties to even), as an object array of Python ints"""
    bits = np.ascontiguousarray(parts, dtype=np.float32).view(np.uint32).astype(np.int64)
    e = (bits >> 23) & 255
    m = np.where(e > 0, (bits & 0x7FFFFF) | 0x800000, bits & 0x7FFFFF)  # |v| = m * 2^(max(e,1) - 150)
    s = np.maximum(e, 1) - 150 - unit_log2                                 # |v| / 2^unit = m * 2^s
    up = m.astype(object) << np.maximum(s, 0).astype(object)
    r = np.clip(-s, 1, 40)
    q, rem, half = m >> r, m & ((np.int64(1) << r) - 1), np.int64(1) << (r - 1)
    down = q + ((rem > half) | ((rem == half) & (q & 1 == 1)))
    mag = np.where(s >= 0, up, down.astype(object))
    return np.where(bits >> 31 == 1, -mag, mag)


def reduce_partials(parts: np.ndarray) -> np.ndarray:
    """float32 partials (..., R) -> the float32 the reduction must return for them (..., )"""
    parts = np.asarray(parts, dtype=np.float32)
    if parts.shape[-1] == 1:
        return parts[..., 0].copy()
    nan = np.isnan(parts).any(-1)
    pinf, ninf = (parts == np.inf).any(-1), (parts == -np.inf).any(-1)
    fin = np.where(np.isfinite(parts), parts, np.float32(0))
    total = round_to_unit(fin).sum(axis=-1)
    out = np.array([to_float32_rne(int(t), UNIT_LOG2) for t in np.ravel(total)], dtype=np.float32).reshape(total.shape)
    out[pinf] = np.inf
    out[ninf] = -np.inf
    out[nan | (pinf & ninf)] = np.nan
    return out


def expected_sums(rtnw, X, p, pixels=None):
    """what a render with params p writes for `pixels` (default: all), from X[s, pixel, channel] = sample s's value"""
    pixels = np.arange(X.shape[1]) if pixels is None else np.asarray(pixels)
    cum = [int(c) for c in rtnw.plan_sample_ranges(p)]
    total = cum[-1]
    out = np.empty((len(pixels), 3), np.float32)
    rotate = bool(p.flags & rtnw.F_ROTATE_SAMPLES)
    groups = {}
    for i, pix in enumerate(pixels):
        m = _pixel_sample_count(p, int(pix))
        b = ((p.sample_begin - int(pix)) % p.sample_stride) if rotate else p.sample_begin
        groups.setdefault((m, b), []).append(i)
    for (m, b), idx in groups.items():
        idx = np.array(idx)
        parts = np.zeros((len(idx), 3, len(cum) - 1), np.float32)
        for c in range(len(cum) - 1):
            acc = np.zeros((len(idx), 3), np.float32)
            for k in range(cum[c] * m // total, cum[c + 1] * m // total):  # k_render: acc starts at 0.f, samples in order
                acc = acc + X[b + k * p.sample_stride, pixels[idx]]
            parts[:, :, c] = acc
        out[idx] = reduce_partials(parts)
    return out


def assert_bits_equal(got, want, what=""):
    """bit for bit, NaN equal to NaN and +0 equal to -0"""
    got, want = np.asarray(got, np.float32).reshape(want.shape), np.asarray(want, np.float32)
    same = (got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want)) | ((got == 0) & (want == 0))
    if not same.all():
        bad = np.argwhere(~same)[:5]
        raise AssertionError(f"{what}: {(~same).sum()} of {same.size} values differ, e.g. at {bad.tolist()}: "
                             f"got {[got[tuple(i)] for i in bad]} want {[want[tuple(i)] for i in bad]}")


# ------------------------------------------------------------------------------------------------ the reference, on the CPU
def test_to_float32_rne_matches_numpy_where_it_rounds_once():
    rng = random.Random(5)
    for _ in range(20000):
        n = rng.randrange(-(1 << 53) + 1, 1 << 53) >> rng.randrange(0, 53)  # exact in a double
        u = rng.randrange(-200, 75)  # below 2^128: the overflow is checked by hand below
        want, got = np.float32(math.ldexp(float(n), u)), to_float32_rne(n, u)
        assert got.view(np.uint32) == want.view(np.uint32), (n, u, got, want)


def test_to_float32_rne_ties_overflow_and_double_rounding():
    t = lambda n, u=0: float(to_float32_rne(n, u))
    assert t((1 << 24) + 1) == 2.0 ** 24 and t((1 << 24) + 3) == 2.0 ** 24 + 4    # halfway: to even
    assert t(-((1 << 24) + 1)) == -(2.0 ** 24) and t((1 << 25) + 2) == 2.0 ** 25  # and a tie one binade up
    n = (((1 << 24) + 1) << 40) + 1                  # just above a tie; a double drops the +1 and then rounds down
    assert t(n) == 2.0 ** 64 + 2.0 ** 41 and float(np.float32(float(n))) == 2.0 ** 64
    assert t(3, -55) == 1.5 * 2.0 ** -54 and t(1, -200) == 0.0 and t(3, -150) == 2.0 ** -148  # below the normal range
    fmax = ((1 << 24) - 1) << 104
    assert t(fmax) == F32_MAX and t(fmax + (1 << 103) - 1) == F32_MAX and t(fmax + (1 << 103)) == math.inf
    assert t(-(fmax + (1 << 103))) == -math.inf and t(1 << 300) == math.inf


def test_round_to_unit_matches_fractions():
    rng = np.random.default_rng(8)
    v = rng.integers(0, 2 ** 32, 20000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    v = v[np.isfinite(v)]
    ties = np.array([0.5, 1.5, 2.5, 3.5, 1 / 3, 1e-30], np.float64) * 2.0 ** -54
    v = np.concatenate([v, ties.astype(np.float32), -ties.astype(np.float32), np.float32([0.0, -0.0, 1e-45, F32_MAX, 0.73])])
    got = round_to_unit(v)
    for x, g in zip(v, got):
        assert g == round(Fraction(float(x)) * 2 ** -UNIT_LOG2), x  # round() of a Fraction: ties to even
    assert list(round_to_unit(np.float32([1.5 * 2.0 ** -54, 2.5 * 2.0 ** -54, -2.5 * 2.0 ** -54]))) == [2, 2, -2]


def test_reduce_partials_specials_and_exactness():
    inf, nan = np.float32(np.inf), np.float32(np.nan)
    r = reduce_partials(np.float32([[1, inf, 2], [inf, -inf, 0], [nan, 1, 1], [-inf, 5, 5], [1e30, -1e30, 1e-13],
                                    [F32_MAX, F32_MAX, 0], [2.0 ** 22, 2.0 ** 22, 2.0 ** 22], [1e-30, 1e-30, 1e-30]]))
    assert r[0] == np.inf and np.isnan(r[1]) and np.isnan(r[2]) and r[3] == -np.inf
    assert r[4] == np.float32(to_float32_rne(round(Fraction(float(np.float32(1e-13))) * 2 ** 54), -54)) and r[4] != 0
    assert r[5] == np.inf and r[6] == np.float32(3 * 2.0 ** 22) and r[7] == 0
    assert reduce_partials(np.float32([[1e-30]]))[0] == np.float32(1e-30)  # one range: the float partial itself


# ------------------------------------------------------------------------------------------------ the magnitude wall
EMISSIONS = [0.0, 1e-30, 2.0 ** -60, 1.5 * 2.0 ** -54, 2.5 * 2.0 ** -54, 0.73, 15.0, 1e5, 2.0 ** 22 - 1, 2.0 ** 22, 3e6, 1e9,
             1e37, F32_MAX, 1e-13, 1e20, math.inf, -math.inf, math.nan]  # neighbours in this list are neighbouring tiles
NX, NY, MAX_NS, SEED = 64, 16, 200, 77


def _wall_desc(rtnw):
    """two rows of 1 x 2 tiles: (e, -e, next e) and (-e, e, previous e), one RTNW_PRIM_RECT_XY diffuse_light per tile at z = 0"""
    hs = rtnw.HostScene("two_perlin")  # borrow the perlin tables / xform identity, as raysets.scene_with_material does
    d = rtnw.SceneDesc()
    C.memmove(C.byref(d), C.byref(hs.desc), C.sizeof(d))
    n, cols = len(EMISSIONS), len(EMISSIONS)
    tex, mat, prim = (rtnw.Texture * (2 * n))(), (rtnw.Material * (2 * n))(), (rtnw.Prim * (2 * n))()
    ids = (C.c_int32 * (2 * n))(*range(2 * n))
    for row in range(2):
        for col in range(cols):
            t = row * cols + col
            e, other = EMISSIONS[col], EMISSIONS[(col + (1 if row == 0 else -1)) % n]
            tex[t].kind = 0
            tex[t].c[0], tex[t].c[1], tex[t].c[2] = (e, -e, other) if row == 0 else (-e, e, other)
            mat[t].kind, mat[t].tex = 3, t
            x0, y0 = col - cols / 2, 2.0 * row - 2.0
            prim[t].f[0], prim[t].f[1], prim[t].f[2], prim[t].f[3], prim[t].f[4] = x0, x0 + 1, y0, y0 + 2, 0.0
            prim[t].kx, prim[t].mat = 2, t
    item = (rtnw.Item * 1)()
    item[0].kind, item[0].first, item[0].count = 0, 0, 2 * n
    item[0].bmin[0], item[0].bmin[1], item[0].bmin[2] = -cols / 2, -2.0, -1e-4
    item[0].bmax[0], item[0].bmax[1], item[0].bmax[2] = cols / 2, 2.0, 1e-4
    d.n_items, d.items, d.n_nodes = 1, item, 0
    d.n_prim_slots, d.prims, d.prim_ids = 2 * n, prim, ids
    d.n_materials, d.materials, d.n_textures, d.textures = 2 * n, mat, 2 * n, tex
    return d, (hs, tex, mat, prim, ids, item)


def _params(rtnw, ns, flags, begin=0, stride=1, ranges=0, pixel_begin=0, pixel_stride=1, pixel_count=0, seed=SEED):
    return rtnw.RenderParams(NX, NY, begin, ns, stride, 50, 0.001, rtnw.FLT_MAX, rtnw.BG_BLACK, rtnw.F_EMIT | flags, seed,
                             pixel_begin, pixel_stride, pixel_count, ranges)


def _samples(render_one, n):
    """X[s, pixel, channel] for s < n, one single-sample render each"""
    return np.stack([render_one(s).reshape(-1, 3) for s in range(n)])


@pytest.fixture(scope="module")
def wall(rtnw, ctx):
    d, keep = _wall_desc(rtnw)
    ds = ctx.upload(d)
    # a view a little larger than the wall (19 x 4 units at 40 units): ~3.1 x 6.2 pixels per tile, tile edges inside pixels
    cam = rtnw.make_camera((0, 0, 40), (0, 0, 0), 2 * math.degrees(math.atan(2.6 / 40)), NX / NY, 0.0, 40.0, 0.0, 1.0)
    X = {}
    for denan in (0, rtnw.F_DE_NAN):
        X[denan] = _samples(lambda s: ds.render(cam, _params(rtnw, 1, denan, begin=s, ranges=1))[0], MAX_NS)
    # the wall must reach every emission: huge, tiny, infinite and NaN samples, and pixels that mix them
    x = X[0]
    assert np.isnan(x).any() and (x == np.inf).any() and (x == -np.inf).any() and (x == np.float32(F32_MAX)).any()
    assert (x == np.float32(1.5 * 2.0 ** -54)).any() and (x == np.float32(1e5)).any() and (x == 0).mean() < 0.5
    assert not np.isnan(X[rtnw.F_DE_NAN]).any() and (X[rtnw.F_DE_NAN] == np.inf).any()
    mixed = (x[:, :, 0] == np.inf).any(0) & (x[:, :, 0] == -np.inf).any(0)
    assert mixed.any(), "no pixel sees both the +inf and the -inf tile"
    yield rtnw, ds, cam, X, keep
    ds.close()


@pytest.mark.gpu
@pytest.mark.parametrize("denan", [False, True])
@pytest.mark.parametrize("ranges", [0, 2, 3, 64, 65])
@pytest.mark.parametrize("ns", [1, 2, 3, 5, 37, 64, 200])
def test_wall_schedules(wall, ns, ranges, denan):
    """every schedule of ranges: the default one (which grows past 4 samples a range above ~110 spp), forced counts, and
    65 (capped to 64)"""
    rtnw, ds, cam, X, _ = wall
    f = rtnw.F_DE_NAN if denan else 0
    p = _params(rtnw, ns, f, ranges=ranges)
    got, st = ds.render(cam, p)
    assert st.sample_ranges == len(rtnw.plan_sample_ranges(p)) - 1 <= 64
    assert_bits_equal(got.reshape(-1, 3), expected_sums(rtnw, X[f], p), f"ns={ns} ranges={ranges} de_nan={denan}")


@pytest.mark.gpu
@pytest.mark.parametrize("ns,world", [(1, 2), (2, 3), (5, 2), (64, 3), (200, 2)])
def test_wall_rotated_samples(wall, ns, world):
    """RTNW_F_ROTATE_SAMPLES (one rank's share of a multi-GPU frame), including ns < G: pixels that own no sample"""
    rtnw, ds, cam, X, _ = wall
    for g in range(world):
        for ranges in (0, 3):
            p = _params(rtnw, ns, rtnw.F_ROTATE_SAMPLES, begin=g, stride=world, ranges=ranges)
            got, _ = ds.render(cam, p)
            assert_bits_equal(got.reshape(-1, 3), expected_sums(rtnw, X[0], p), f"rank {g} of {world}, ns={ns}")


@pytest.mark.gpu
@pytest.mark.parametrize("fast", [False, True])
def test_wall_entry_points_and_accumulated_subset(wall, fast):
    """rtnw_render and rtnw_render_device agree with the reference with and without RTNW_F_FAST_BVH; a pixel subset with
    RTNW_F_ACCUMULATE adds the reduced value to a prefilled buffer (+-inf and NaN among the prefill) and leaves the other
    pixels alone"""
    import torch
    rtnw, ds, cam, X, _ = wall
    f = rtnw.F_FAST_BVH if fast else 0
    for ns in (37, 64):
        p = _params(rtnw, ns, f)
        want = expected_sums(rtnw, X[0], p)
        got, _ = ds.render(cam, p)
        assert_bits_equal(got.reshape(-1, 3), want, "rtnw_render")
        buf = torch.full((NY, NX, 3), 3.0, dtype=torch.float32, device="cuda")
        ds.render_device(cam, p, buf.data_ptr())
        assert_bits_equal(buf.cpu().numpy().reshape(-1, 3), want, "rtnw_render_device")
        rng = np.random.default_rng(ns)
        pre = (rng.standard_normal((NY * NX, 3)) * 10.0 ** rng.integers(-20, 30, (NY * NX, 1))).astype(np.float32)
        pre[::7, 0], pre[::11, 1], pre[::13, 2] = np.inf, -np.inf, np.nan
        buf = torch.from_numpy(pre.reshape(NY, NX, 3).copy()).cuda()
        begin, stride, count = 3, 5, (NY * NX - 3) // 5
        ps = _params(rtnw, ns, f | rtnw.F_ACCUMULATE, pixel_begin=begin, pixel_stride=stride, pixel_count=count)
        ds.render_device(cam, ps, buf.data_ptr())
        idx = begin + stride * np.arange(count)
        want_acc = pre.copy()
        want_acc[idx] = pre[idx] + expected_sums(rtnw, X[0], ps, idx)
        assert_bits_equal(buf.cpu().numpy().reshape(-1, 3), want_acc, "accumulated pixel subset")


@pytest.mark.gpu
@pytest.mark.parametrize("devs", [[0, 0], [0, 0, 0]])
def test_wall_multi_device(wall, devs):
    """rtnw_render_multi and the colour of rtnw_render_aov_multi: each rank's share reduced exactly, the shares added in
    rank order in float32 (one device listed several times: the same code path as several GPUs)"""
    rtnw, _, cam, X, _ = wall
    d, keep_desc = _wall_desc(rtnw)
    mc = rtnw.MultiContext(devs)
    ms = mc.upload(d)
    try:
        for ns in (2, 37, 64):
            p = _params(rtnw, ns, 0)
            n = len(devs)
            want = None
            for g in range(n):
                share = expected_sums(rtnw, X[0], _params(rtnw, ns, rtnw.F_ROTATE_SAMPLES, begin=g, stride=n))
                want = share if want is None else want + share
            got, _ = ms.render(cam, p)
            assert_bits_equal(got.reshape(-1, 3), want, f"rtnw_render_multi {devs} ns={ns}")
            sums, _, _, _ = ms.render_aov(cam, p)
            assert_bits_equal(sums.reshape(-1, 3), want, f"rtnw_render_aov_multi {devs} ns={ns}")
    finally:
        ms.close()
        mc.close()


@pytest.mark.gpu
def test_wall_is_deterministic_and_leaves_the_plane_clean(rtnw, ctx, wall):
    """two renders of the wall are byte-identical, and an ordinary render on the same pixels afterwards equals one on a
    fresh context: no flag or residue is left in the accumulation plane"""
    _, ds, cam, _, _ = wall
    p = _params(rtnw, 64, 0)
    a, _ = ds.render(cam, p)
    b, _ = ds.render(cam, p)
    assert a.tobytes() == b.tobytes()
    hs = rtnw.HostScene("cornell_box")
    hcam, hp = hs.camera(NX, NY), hs.params(nx=NX, ny=NY, ns=16, seed=5)
    bs = ctx.upload(hs.desc_ptr)
    after, _ = bs.render(hcam, hp)
    bs.close()
    fresh = rtnw.Context(0)
    fs = fresh.upload(hs.desc_ptr)
    clean, _ = fs.render(hcam, hp)
    fs.close()
    fresh.close()
    assert after.tobytes() == clean.tobytes()


# ------------------------------------------------------------------------------------------------ real scenes
@pytest.mark.gpu
@pytest.mark.parametrize("lights", [False, True])
@pytest.mark.parametrize("name", ["cornell_box", "cornell_smoke"])
def test_real_scenes(rtnw, ctx, name, lights):
    """the Cornell scenes at 256 spp, with and without RTNW_F_LIGHT_SAMPLING (whose path weights are heavy-tailed)"""
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    nx = ny = 24
    ns, f = 256, rtnw.F_LIGHT_SAMPLING if lights else 0
    cam = hs.camera(nx, ny)
    X = _samples(lambda s: ds.render(cam, hs.params(nx=nx, ny=ny, ns=1, seed=9, sample_begin=s, sample_ranges=1,
                                                    flags_extra=f))[0], ns)
    p = hs.params(nx=nx, ny=ny, ns=ns, seed=9, flags_extra=f)
    got, st = ds.render(cam, p)
    assert st.sample_ranges > 1
    assert_bits_equal(got.reshape(-1, 3), expected_sums(rtnw, X, p), f"{name} lights={lights}")
    ds.close()
