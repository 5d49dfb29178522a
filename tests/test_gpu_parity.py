"""GPU parity tests: the CUDA path (through the C-ABI of include/rtnw.h) against the reference renderer itself
(oracle/_ref/libref_oracle.so = the reference's headers compiled unmodified + the F2 aabb fix, SURVEY.md §8c).

Bars (BASELINE.json north_star): closest-hit leaf ids and box faces bit-exact; t / p / normal bit-exact (float32, no
FMA contraction on either side); u,v within 1e-5 (libm atan2f/asinf); images compared sample for sample because the
reference is driven by the same Philox stream as the GPU (oracle/ref_harness.cpp hook).
"""
import numpy as np
import pytest

import oracle_port as op
import ref_oracle as ro
from raysets import FLT_MAX, assert_hits_equal, make_rays, reference_camera_rays, reference_scene, scene_with_material

# the reference side is the compiled reference when it is built, else the C restatement pinned bit-exact to it (raysets.py)
pytestmark = pytest.mark.gpu

TRACE_SCENES = ["ch01_random", "two_perlin", "cornell_box", "cornell_smoke", "final", "final+bvh", "final_northstar", "earth",
                "simple_light", "cornell_smoke+bvh", "random_scene", "random_scene+bvh", "test"]


@pytest.mark.parametrize("name", TRACE_SCENES)
def test_closest_hit_ids_bit_exact(rtnw, ctx, name):
    rs, rays = make_rays(name, rtnw=rtnw)
    want = rs.trace(rays, 0.001, FLT_MAX, seed=11)
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    got = ds.trace(rays, 0.001, FLT_MAX, flags=0, seed=11)
    assert (want["prim_id"] >= 0).sum() > len(rays) // 10
    assert_hits_equal(got, want)
    # mat_id is this framework's table index: check it names the same material kind the reference hit
    ds.close()


@pytest.mark.parametrize("name", ["final+bvh", "final_northstar", "ch01_random+bvh", "cornell_smoke+bvh", "random_scene+bvh"])
def test_fast_bvh_mode_finds_the_same_closest_hit_with_fewer_tests(rtnw, ctx, name):
    """RTNW_F_FAST_BVH: a SAH tree over the LEAVES' own boxes instead of the reference's leaf-parent gates, plain list elements
    first, BVH elements two at a time, boxes and leaves tested against the running closest hit instead of the reference's
    un-narrowed range.  Gate (VERDICT r1 item 6): on >= 1e6 rays per scene the closest hit is the exact mode's - same t bit for
    bit, and the same leaf except among candidates of EQUAL t (a documented tie: the exact mode lets the later leaf win, the
    fast mode may have culled it) - with fewer primitive tests and fewer tests in total."""
    rng = np.random.default_rng(17)
    rs, base = make_rays(name, n_primary=3000, seed=5, rtnw=rtnw)
    reps = -(-1_000_000 // len(base))
    rays = np.tile(base, reps)
    jitter = (1.0 + 1e-3 * rng.standard_normal((len(rays), 3))).astype(np.float32)
    rays["direction"] = rays["direction"] * jitter  # distinct rays around the deterministic set (the first copy stays exact)
    rays["direction"][:len(base)] = base["direction"]
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    exact = ds.trace(rays, 0.001, FLT_MAX, flags=0, seed=3)
    fast = ds.trace(rays, 0.001, FLT_MAX, flags=rtnw.F_FAST_BVH, seed=3)
    assert_hits_equal(exact[:len(base)], rs.trace(base, 0.001, FLT_MAX, seed=3))
    hit = exact["prim_id"] >= 0
    assert np.array_equal(fast["prim_id"] >= 0, hit)
    same_t = fast["t"][hit].view(np.uint32) == exact["t"][hit].view(np.uint32)
    nan_t = np.isnan(fast["t"][hit]) | np.isnan(exact["t"][hit])
    assert (same_t | nan_t).all(), f"{(~(same_t | nan_t)).sum()} closest hits differ in t"
    other = fast["prim_id"][hit] != exact["prim_id"][hit]
    assert other.mean() < 0.05, f"{other.mean():.4f} of the hits resolve an equal-t tie differently"
    nx, ny = 160, 120
    cam = hs.camera(nx, ny)
    a, sa = ds.render(cam, hs.params(nx=nx, ny=ny, ns=8, seed=2, flags_extra=rtnw.F_COUNTERS))
    b, sb = ds.render(cam, hs.params(nx=nx, ny=ny, ns=8, seed=2, flags_extra=rtnw.F_COUNTERS | rtnw.F_FAST_BVH))
    # one more level of boxes (each leaf behind its own box), fewer primitive tests, fewer tests in total
    assert sb.prim_tests < sa.prim_tests and sb.box_tests + sb.prim_tests < sa.box_tests + sa.prim_tests
    ok = np.isfinite(a).all(axis=2) & np.isfinite(b).all(axis=2)
    assert np.isclose(a[ok], b[ok], rtol=1e-4, atol=1e-5).all(axis=1).mean() > 0.97  # a tie resolved differently changes a path
    assert abs(a[ok].sum() - b[ok].sum()) < 0.01 * a[ok].sum()
    ds.close()


def test_trace_t_range_and_empty_input(rtnw, ctx):
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    assert len(ds.trace(np.zeros(0, dtype=rtnw.RAY_DTYPE))) == 0
    rs, rays = make_rays("cornell_box", n_primary=500, rtnw=rtnw)
    for t_min, t_max in [(0.0, FLT_MAX), (0.01, 900.0), (100.0, 700.0)]:
        assert_hits_equal(ds.trace(rays, t_min, t_max, seed=2), rs.trace(rays, t_min, t_max, seed=2))
    ds.close()


def test_camera_rays_bit_exact(rtnw, ctx):
    rng = np.random.default_rng(1)
    for name, nx, ny in [("ch01_random", 200, 100), ("final", 1000, 1000), ("two_perlin", 400, 200)]:
        n = 4000
        ij = np.stack([rng.integers(0, nx, n), rng.integers(0, ny, n)], axis=1)
        s = rng.integers(0, 1000, n)
        want = reference_camera_rays(rtnw, name, nx, ny, ij, s, seed=99)
        cam = rtnw.HostScene(name).camera(nx, ny)
        got = rtnw.camera_rays(ctx, cam, nx, ny, ij, s, seed=99)
        for f in ("origin", "direction", "time", "key"):
            assert np.array_equal(got[f], want[f]), f


def test_perlin_and_textures(rtnw, ctx):
    rng = np.random.default_rng(2)
    hs = rtnw.HostScene("two_perlin")
    live = ro.available()
    if live:
        ro.RefScene("two_perlin", tagged=False)  # same perlin tables in the reference's statics
    ds = ctx.upload(hs.desc_ptr)
    xyz = np.concatenate([rng.normal(scale=3, size=(3000, 3)), rng.normal(scale=400, size=(3000, 3)),
                          rng.integers(-5, 5, size=(500, 3)).astype(np.float64)]).astype(np.float32)
    for which in (0, 1):
        got = ds.eval_perlin(which, xyz)
        want = ro.eval_perlin(which, xyz) if live else op.eval_perlin(rtnw, hs.desc_ptr, which, xyz)
        assert np.array_equal(got, want), f"perlin which={which}: {np.abs(got - want).max()}"
    uvp = np.concatenate([rng.random((len(xyz), 2)).astype(np.float32), xyz], axis=1)
    # textures of two_perlin: 0 = checker(even 1, odd 2), 3 = noise(4)
    d = hs.desc
    kinds = [d.textures[i].kind for i in range(d.n_textures)]
    checker, noise = kinds.index(1), kinds.index(2)
    got = ds.eval_texture(checker, uvp)
    want = ro.eval_texture(1, [0.2, 0.3, 0.1, 0.9, 0.9, 0.9], uvp) if live else op.eval_texture(rtnw, hs.desc_ptr, checker, uvp)
    assert (np.all(got == want, axis=1)).mean() > 0.999  # sign of a product of three sinf near zero may flip by an ulp
    got = ds.eval_texture(noise, uvp)
    want = ro.eval_texture(2, [4.0], uvp) if live else op.eval_texture(rtnw, hs.desc_ptr, noise, uvp)
    assert np.allclose(got, want, rtol=0, atol=2e-6), np.abs(got - want).max()
    ds.close()
    hs = rtnw.HostScene("earth")
    ds = ctx.upload(hs.desc_ptr)
    d = hs.desc
    img = [d.textures[i].kind for i in range(d.n_textures)].index(3)
    uvp[:50, :2] = np.array([[0, 0], [1, 1], [0, 1], [1, 0], [0.5, 0.5]] * 10, dtype=np.float32)
    assert np.array_equal(ds.eval_texture(img, uvp), ro.eval_texture(3, [], uvp) if live else op.eval_texture(rtnw, hs.desc_ptr, img, uvp))
    ds.close()


@pytest.mark.parametrize("kind,rgb,f,scale", [(0, (0.4, 0.2, 0.1), 0, 0), (0, (0, 0, 0), 0, 4.0), (1, (0.8, 0.8, 0.9), 0.3, 0),
                                              (1, (1, 1, 1), 0.0, 0), (2, (0, 0, 0), 1.5, 0), (2, (0, 0, 0), 2.5, 0),
                                              (3, (7, 7, 7), 0, 0), (4, (0.2, 0.4, 0.9), 0, 0)])
def test_scatter_and_emitted_same_stream(rtnw, ctx, kind, rgb, f, scale):
    rng = np.random.default_rng(kind * 10 + int(f * 10))
    n = 4000
    d, keep = scene_with_material(rtnw, kind, rgb, f, scale)
    live = ro.available()
    if live:
        ro.RefScene("two_perlin", tagged=False)
    ds = ctx.upload(d)
    rays = np.zeros(n, dtype=rtnw.RAY_DTYPE)
    rays["origin"] = rng.normal(size=(n, 3))
    rays["direction"] = rng.normal(size=(n, 3)) * rng.choice([0.1, 1.0, 10.0], (n, 1))
    rays["time"] = rng.random(n)
    hits = np.zeros(n, dtype=rtnw.HIT_DTYPE)
    nrm = rng.normal(size=(n, 3))
    hits["normal"] = nrm / np.linalg.norm(nrm, axis=1, keepdims=True)
    hits["p"] = rng.normal(scale=3, size=(n, 3))
    hits["t"] = 1.0
    hits["u"], hits["v"] = rng.random(n), rng.random(n)
    mat = np.tile(np.array([kind, 2 if scale else 0, rgb[0], rgb[1], rgb[2], f, scale, 0], dtype=np.float32), (n, 1))
    w_sc, w_att, w_em, w_flag = ro.scatter(mat, rays, hits, seed=5) if live else op.scatter(rtnw, d, rays, hits, seed=5)
    g_sc, g_att, g_em, g_flag = ds.scatter(rays, hits, seed=5)
    assert np.array_equal(g_flag, w_flag)
    assert np.array_equal(g_em, w_em)
    if scale:
        assert np.allclose(g_att, w_att, rtol=0, atol=2e-6)
    else:
        assert np.array_equal(g_att, w_att)
    for fld in ("origin", "time"):
        assert np.array_equal(g_sc[fld], w_sc[fld]), fld
    a, b = g_sc["direction"], w_sc["direction"]
    if kind == 2:
        # schlick() goes through pow() in double on the CPU; a last-bit difference can flip reflect/refract for a draw
        # that lands within an ulp of reflect_prob.  NaN directions (sqrt of a negative, PSC/material.h:103) must agree.
        same = np.all((a == b) | (np.isnan(a) & np.isnan(b)), axis=1)
        assert same.mean() > 0.999
    else:
        assert np.array_equal(a, b)
    ds.close()


RENDER_CASES = [("ch01_random", 64, 32, 6), ("two_perlin", 64, 32, 6), ("cornell_box", 48, 48, 8), ("cornell_smoke", 48, 48, 8),
                ("final", 40, 40, 4), ("final+bvh", 40, 40, 4), ("final_northstar", 40, 40, 4), ("simple_light", 48, 24, 6),
                ("earth", 40, 40, 4), ("random_scene", 64, 32, 6), ("test", 48, 24, 6)]


# every BASELINE.json config at its STATED image size (spp reduced to what the single-threaded reference renders in seconds):
# the same per-path streams on both sides, so each of the 10^5..10^6 pixels is compared with the reference's own pixel
FULL_SIZE_CASES = [("ch01_random", 200, 100, 2), ("two_perlin", 400, 200, 2), ("cornell_box", 500, 500, 1),
                   ("cornell_smoke", 500, 500, 1), ("final+bvh", 1000, 1000, 1), ("final_northstar", 1000, 1000, 1)]


@pytest.mark.parametrize("name,nx,ny,ns", RENDER_CASES + FULL_SIZE_CASES)
def test_render_matches_reference_sample_for_sample(rtnw, ctx, name, nx, ny, ns):
    """Same Philox stream on both sides => the per-pixel SUMS agree except where a libm ulp flips a branch.
    Tolerance: >= 99% of pixels within 2e-5 relative (+1e-6 absolute) and total radiance within 0.2%.
    Documented deviation: the GPU multiplies attenuations front to back (iterative color()), the reference back to
    front (recursion), which reassociates a product of <= 51 floats."""
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    cam = hs.camera(nx, ny)
    p = hs.params(nx=nx, ny=ny, ns=ns, seed=1234)
    got, st = ds.render(cam, p)
    rs = reference_scene(rtnw, name)
    want, rst = rs.render(nx, ny, ns, seed=1234, rng_mode=1)
    assert st.paths == nx * ny * ns
    close = np.isclose(got, want, rtol=2e-5, atol=1e-6).all(axis=2)
    assert close.mean() >= 0.99, f"{name}: only {close.mean():.4f} of pixels agree"
    assert abs(got.sum() - want.sum()) <= 2e-3 * abs(want.sum()) + 1e-3
    # the two sides must also agree on how many closest-hit queries the paths needed
    assert abs(st.rays - rst["rays"]) <= 0.002 * rst["rays"], (st.rays, rst["rays"])
    ds.close()


def test_gpu_tests_exactly_the_primitives_the_reference_tests(rtnw, ctx):
    """RTNW_F_COUNTERS.  The gate tree (DESIGN.md §3) replaces the reference's hierarchy above the leaves' parent boxes, so
    the GPU does FEWER box tests than the reference's bvh_node::hit, but it must hand the ray to exactly the same leaves:
    the number of primitive hit() calls equals the reference restatement's count."""
    import oracle_port as op
    for name, nx, ny, ns in [("final+bvh", 32, 32, 2), ("final_northstar", 32, 32, 2), ("ch01_random+bvh", 32, 16, 2)]:
        hs = rtnw.HostScene(name)
        ds = ctx.upload(hs.desc_ptr)
        p = hs.params(nx=nx, ny=ny, ns=ns, seed=9, flags_extra=rtnw.F_COUNTERS)
        _, st = ds.render(hs.camera(nx, ny), p)
        _, ost = op.render(rtnw, hs.desc_ptr, hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=9))
        assert abs(st.rays - ost["rays"]) <= 0.003 * ost["rays"]
        assert abs(st.prim_tests - ost["prim_tests"]) <= 0.004 * ost["prim_tests"], (name, st.prim_tests, ost["prim_tests"])
        assert 0 < st.box_tests < ost["box_tests"], (name, st.box_tests, ost["box_tests"])
        ds.close()


def test_sample_split_is_a_partition(rtnw, ctx):
    """multi-GPU split (rank g renders samples g, g+G, ...): the union equals the single render up to float order"""
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    nx = ny = 64
    cam = hs.camera(nx, ny)
    full, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=8, seed=5))
    again, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=8, seed=5))
    assert np.array_equal(full, again)  # deterministic: no atomics on the image
    parts = sum(ds.render(cam, hs.params(nx=nx, ny=ny, ns=2, seed=5, sample_begin=g, sample_stride=4))[0].astype(np.float64)
                for g in range(4))
    assert np.allclose(parts, full, rtol=1e-5, atol=1e-6)
    other, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=8, seed=6))
    assert not np.array_equal(full, other)
    ds.close()


def test_full_size_render_properties(rtnw, ctx):
    """BASELINE config 5 at full resolution (1000x1000), reduced spp: size-independent properties."""
    hs = rtnw.HostScene("final_northstar")
    ds = ctx.upload(hs.desc_ptr)
    nx = ny = 1000
    cam = hs.camera(nx, ny)
    a, st = ds.render(cam, hs.params(nx=nx, ny=ny, ns=4, seed=1))
    assert st.paths == 4_000_000 and 2.0 < st.rays / st.paths < 6.0
    assert np.isfinite(a).all() and (a >= 0).all()
    # additivity over the sample partition
    b = ds.render(cam, hs.params(nx=nx, ny=ny, ns=2, seed=1, sample_begin=0, sample_stride=2))[0].astype(np.float64) + \
        ds.render(cam, hs.params(nx=nx, ny=ny, ns=2, seed=1, sample_begin=1, sample_stride=2))[0].astype(np.float64)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-6)
    # the fast traversal mode renders the same image up to equal-t ties (adjacent floor boxes share face planes)
    c, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=4, seed=1, flags_extra=rtnw.F_FAST_BVH))
    assert (np.isclose(a, c, rtol=1e-5, atol=1e-6).all(axis=2)).mean() > 0.97 and abs(c.sum() - a.sum()) < 0.01 * a.sum()
    # coarse known-answer: the light (7,7,7) is visible and the mean is in the range of the shipped final renders
    q = rtnw.quantize(a, 4)
    assert q.shape == (ny, nx, 3) and q.max() == 255 and 15 < q.mean() < 80
    ds.close()


def test_errors_do_not_cross_the_boundary(rtnw, ctx):
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    cam = hs.camera(8, 8)
    with pytest.raises(rtnw.RtnwError) as e:
        ds.render(cam, hs.params(nx=8, ny=8, ns=0))
    assert e.value.code == rtnw.RTNW_ERR_INVALID
    import ctypes as C
    bad = rtnw.SceneDesc()
    C.memmove(C.byref(bad), C.byref(hs.desc), C.sizeof(bad))
    bad.abi_version = 3
    with pytest.raises(rtnw.RtnwError):
        ctx.upload(bad)
    ds.close()


def test_gate_queue_throttle_and_wrap_under_stress(rtnw, ctx):
    """600 nested shells in one bvh_node: a ray towards the centre passes every gate, so a block's 256 rays queue far
    more gates than the 4096-entry ring holds — node work must pause, the ring must wrap, and the result must still be
    the reference's (checked against the C restatement, which is pinned to the compiled reference)."""
    import oracle_port as op
    hs = rtnw.HostScene("stress_shells+bvh")
    ds = ctx.upload(hs.desc_ptr)
    rng = np.random.default_rng(3)
    n = 3000
    rays = np.zeros(n, dtype=rtnw.RAY_DTYPE)
    o = rng.normal(size=(n, 3)); o = 12.0 * o / np.linalg.norm(o, axis=1, keepdims=True)
    rays["origin"] = o
    rays["direction"] = -o + rng.normal(scale=0.3, size=(n, 3))
    rays["origin"][n // 2:] = rng.normal(scale=2.0, size=(n - n // 2, 3))  # origins between the shells
    rays["time"] = rng.random(n)
    want = op.trace(rtnw, hs.desc_ptr, rays, 0.001, FLT_MAX, seed=4)
    assert (want["prim_id"] >= 0).mean() > 0.9
    assert_hits_equal(ds.trace(rays, 0.001, FLT_MAX, seed=4), want)
    nx, ny, ns = 64, 32, 3
    got, st = ds.render(hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=8, flags_extra=rtnw.F_COUNTERS))
    ref, ost = op.render(rtnw, hs.desc_ptr, hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=8))
    assert np.isclose(got, ref, rtol=2e-5, atol=1e-6).all(axis=2).mean() >= 0.99
    assert abs(st.prim_tests - ost["prim_tests"]) <= 0.004 * ost["prim_tests"]
    ds.close()


@pytest.mark.parametrize("name,n,ns,reps", [("final_northstar", 160, 6, 2), ("final+bvh", 160, 6, 2), ("stress_shells+bvh", 160, 6, 2),
                                            ("final_northstar", 1000, 4, 150), ("final+bvh", 1000, 4, 60)])
def test_render_is_bitwise_deterministic(rtnw, ctx, name, n, ns, reps):
    """No atomics on the image and an order-independent closest-hit key: repeated runs must agree bit for bit, whatever
    order the block's threads happened to take the shared-memory tasks in (stands in for racecheck, closed on this pool).
    The full-size soak is the regression test of a real race: the children a round pushes reuse the stack slots the round
    pops, and about once in 10^8 warp-rounds a starved warp read its task after another warp's push had overwritten it — one
    wrong path in ~7 % of 1000x1000 frames, invisible at small sizes (fixed by the node-warp barrier)."""
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    nx = ny = n
    cam = hs.camera(nx, ny)
    a, sa = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=77))
    for rep in range(reps):
        b, sb = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=77))
        diff = (a.view(np.uint32) != b.view(np.uint32)).any(axis=2)
        assert not diff.any() and sa.rays == sb.rays, (f"repetition {rep}: {int(diff.sum())} pixels differ (first "
                                                       f"{np.argwhere(diff)[:4].tolist()}), rays {sa.rays} vs {sb.rays}")
    ds.close()


def test_pixel_subset_and_accumulate(rtnw, ctx):
    """rtnw_render_params.pixel_begin/stride/count + RTNW_F_ACCUMULATE (the multi-GPU split of left-over samples): rendering
    7 samples as 3 (all pixels) + 4 (two interleaved pixel subsets, accumulated) reproduces the one-shot render."""
    import torch
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    nx = ny = 48
    cam = hs.camera(nx, ny)
    full, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=7, seed=21))
    acc = torch.full((ny, nx, 3), 123.0, dtype=torch.float32, device="cuda")
    st = ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=3, seed=21), acc.data_ptr())
    assert st.paths == nx * ny * 3
    for r in range(2):
        cnt = len(range(r, nx * ny, 2))
        st = ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=4, seed=21, sample_begin=3, pixel_begin=r, pixel_stride=2, pixel_count=cnt,
                                             flags_extra=rtnw.F_ACCUMULATE), acc.data_ptr())
        assert st.paths == cnt * 4
    assert np.allclose(acc.cpu().numpy(), full, rtol=1e-6, atol=1e-6)
    with pytest.raises(rtnw.RtnwError):  # subsets are a device-buffer feature
        ds.render(cam, hs.params(nx=nx, ny=ny, ns=1, pixel_begin=0, pixel_stride=2, pixel_count=10))
    with pytest.raises(rtnw.RtnwError):
        ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=1, pixel_begin=5, pixel_stride=1, pixel_count=nx * ny), acc.data_ptr())
    ds.close()


@pytest.mark.parametrize("ns,world", [(7, 3), (10, 8), (3, 8), (12, 4)])
def test_rotated_sample_split_is_an_even_partition(rtnw, ctx, ns, world):
    """RTNW_F_ROTATE_SAMPLES (the multi-GPU split): the ranks' renders sum to the single render for any ns, including
    ns < world (pixels that own no sample on a rank), and every rank traces the same number of paths +- npix % world."""
    import oracle_port as op
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    nx, ny = 40, 30
    cam = hs.camera(nx, ny)
    full, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=33))
    total = np.zeros_like(full, dtype=np.float64)
    paths = []
    for g in range(world):
        p = hs.params(nx=nx, ny=ny, ns=ns, seed=33, sample_begin=g, sample_stride=world, flags_extra=rtnw.F_ROTATE_SAMPLES)
        part, st = ds.render(cam, p)
        ref, ost = op.render(rtnw, hs.desc_ptr, cam, p)
        assert st.paths == ost["paths"]
        assert np.isclose(part, ref, rtol=2e-5, atol=1e-6).all(axis=2).mean() >= 0.99
        total += part
        paths.append(st.paths)
    assert sum(paths) == nx * ny * ns and max(paths) - min(paths) <= nx * ny % world + world
    assert np.allclose(total, full, rtol=1e-5, atol=1e-6)
    ds.close()


def test_small_image_sample_ranges(rtnw, ctx):
    """A pixel with enough samples is rendered as several (sample range, pixel) work items whose partial sums are added
    exactly in fixed point: same paths, same rays, the sums equal up to float rounding, and still bitwise reproducible.
    rtnw_render_params.sample_ranges forces the number of ranges (1 = one thread per pixel)."""
    import torch
    hs = rtnw.HostScene("cornell_smoke")
    ds = ctx.upload(hs.desc_ptr)
    nx, ny, ns = 64, 48, 37
    cam = hs.camera(nx, ny)
    one, s1 = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=4, sample_ranges=1))
    assert s1.kernel_launches == 1
    for forced in (0, 5, 64):
        a, sa = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=4, sample_ranges=forced))
        b, sb = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=4, sample_ranges=forced))
        assert sa.kernel_launches == 2 and sa.paths == s1.paths and sa.rays == s1.rays == sb.rays
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert np.allclose(a, one, rtol=1e-5, atol=1e-6)
    # with the multi-GPU split and accumulation on top
    acc = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
    for g in range(2):
        ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=4, sample_begin=g, sample_stride=2, sample_ranges=3,
                                        flags_extra=rtnw.F_ROTATE_SAMPLES | rtnw.F_ACCUMULATE), acc.data_ptr())
    assert np.allclose(acc.cpu().numpy(), one, rtol=1e-5, atol=1e-6)
    ds.close()


def test_fixed_point_range_sums_keep_nan_and_pixel_subsets(rtnw, ctx):
    """the fixed-point plane: a NaN sample (no de_nan) makes its pixel NaN as `col += temp` does; pixels outside a subset
    stay untouched; the plane is clean again for the next render"""
    import torch
    hs = rtnw.HostScene("ch01_random")  # dielectrics, de_nan off in this chapter's view
    ds = ctx.upload(hs.desc_ptr)
    nx, ny, ns = 96, 48, 64
    cam = hs.camera(nx, ny)
    one, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=11, sample_ranges=1))
    many, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=11))
    assert np.array_equal(np.isnan(one), np.isnan(many))
    ok = ~np.isnan(one)
    assert np.allclose(many[ok], one[ok], rtol=1e-5, atol=1e-6)
    acc = torch.full((ny, nx, 3), -7.0, dtype=torch.float32, device="cuda")
    ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=11, pixel_begin=5, pixel_stride=3, pixel_count=400), acc.data_ptr())
    sub = acc.cpu().numpy().reshape(-1, 3)
    idx = 5 + 3 * np.arange(400)
    mask = np.zeros(nx * ny, bool); mask[idx] = True
    assert np.all(sub[~mask] == -7.0)
    ref = many.reshape(-1, 3)[idx]
    assert np.array_equal(np.nan_to_num(sub[idx], nan=-1).view(np.uint32), np.nan_to_num(ref, nan=-1).view(np.uint32))
    again, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=11))
    assert np.array_equal(np.nan_to_num(again, nan=-1).view(np.uint32), np.nan_to_num(many, nan=-1).view(np.uint32))
    ds.close()


def test_device_epilogue_equals_host_epilogue(rtnw, ctx):
    """rtnw_quantize_device (gamma + quantise + clamp on the GPU, after the reduce) is bit-identical to the host epilogue
    rtnw_host_quantize, which restates PSC/main.cpp:315-325; includes values > 1 (light), 0, and every sum the sample-range
    reduction can return: negatives, NaN, +-inf, -0 and means so large that 255.99*sqrt(mean) leaves the int range."""
    import torch
    hs = rtnw.HostScene("cornell_box")
    ds = ctx.upload(hs.desc_ptr)
    nx, ny, ns = 64, 48, 10
    acc = torch.empty(ny, nx, 3, dtype=torch.float32, device="cuda")
    ds.render_device(hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=3), acc.data_ptr())
    sums = acc.cpu().numpy()
    for clamp in (True, False):
        assert np.array_equal(ctx.quantize_device(acc.data_ptr(), nx, ny, ns, clamp), rtnw.quantize(sums, ns, clamp))
    rng = np.random.default_rng(0)
    synth = (rng.random((ny, nx, 3)) * rng.choice([0.0, 1.0, 50.0, 4000.0], (ny, nx, 1))).astype(np.float32)
    t = torch.from_numpy(synth).cuda()
    for n in (1, 3, 100, 1000):
        assert np.array_equal(ctx.quantize_device(t.data_ptr(), nx, ny, n, True), rtnw.quantize(synth, n, True))
    special = np.float32([np.nan, np.inf, -np.inf, -0.0, -1.0, -1e-30, -3e38, 1e20, 7.0377e13, 7.0379e13, 3.4e38, 1e-45])
    synth = (rng.standard_normal((ny, nx, 3)) * 10.0 ** rng.integers(-30, 37, (ny, nx, 3))).astype(np.float32)
    synth.reshape(-1)[:special.size * 50] = np.tile(special, 50)
    t = torch.from_numpy(synth).cuda()
    for n in (1, 3, 100, 1000):
        for clamp in (True, False):
            want = rtnw.quantize(synth, n, clamp)
            assert np.array_equal(ctx.quantize_device(t.data_ptr(), nx, ny, n, clamp), want)
    assert (want == np.int32(-2 ** 31)).any()  # NaN and out-of-range means did reach the x86 conversion result
    ds.close()


def test_adjacent_bvh_items(rtnw, ctx):
    """two bvh_nodes that are neighbours in the top-level list (fixture `twin_bvh`): the cooperative traversal enters a BVH
    item straight after leaving one, with no barrier in between (ADVICE r1: the queue state must not be reset under a
    thread that is still reading it).  Checked against the C restatement of the reference, repeatedly."""
    import oracle_port as op
    hs = rtnw.HostScene("twin_bvh")
    ds = ctx.upload(hs.desc_ptr)
    nx, ny = 200, 100
    cam = hs.camera(nx, ny)
    rng = np.random.default_rng(3)
    ij = np.stack([rng.integers(0, nx, 20000), rng.integers(0, ny, 20000)], axis=1)
    rays = rtnw.camera_rays(ctx, cam, nx, ny, ij, rng.integers(0, 9, 20000), seed=5)
    want = op.trace(rtnw, hs.desc_ptr, rays, seed=5)
    assert (want["prim_id"] >= 0).mean() > 0.3
    for _ in range(5):
        assert_hits_equal(ds.trace(rays, seed=5), want)
    a, sa = ds.render(cam, hs.params(nx=nx, ny=ny, ns=16, seed=9))
    for _ in range(3):
        b, sb = ds.render(cam, hs.params(nx=nx, ny=ny, ns=16, seed=9))
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and sa.rays == sb.rays
    small, _ = op.render(rtnw, hs.desc_ptr, hs.camera(64, 32), hs.params(nx=64, ny=32, ns=4, seed=9))
    got, _ = ds.render(hs.camera(64, 32), hs.params(nx=64, ny=32, ns=4, seed=9))
    assert np.isclose(got, small, rtol=2e-5, atol=1e-6).all(axis=2).mean() > 0.99
    ds.close()


def test_multi_gpu_through_the_c_abi(rtnw, ctx):
    """rtnw_ctx_create_multi / rtnw_render_multi: N devices in one process — the samples of every pixel split over the
    devices, summed on device 0 — equals the one-device render up to float summation order, for even and odd ns.  On a
    one-GPU box the same device is listed twice (two contexts, same code path); with >= 2 GPUs also [0, 1]."""
    hs = rtnw.HostScene("final_northstar")
    nx, ny = 160, 120
    cam = hs.camera(nx, ny)
    ds = ctx.upload(hs.desc_ptr)
    lists = [[0, 0], [0, 0, 0]] + ([[0, 1]] if rtnw.device_count() >= 2 else [])
    for ns in (16, 7):
        one, s1 = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21))
        for devs in lists:
            mc = rtnw.MultiContext(devs)
            ms = mc.upload(hs.desc_ptr)
            a, sa = ms.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21))
            b, sb = ms.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21))
            assert sa.paths == s1.paths == nx * ny * ns and sa.rays == s1.rays
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
            assert np.allclose(a, one, rtol=1e-5, atol=1e-6)
            assert sa.kernel_launches >= len(devs) + 1 and sa.total_ms >= sa.kernel_ms > 0
            with pytest.raises(rtnw.RtnwError):
                ms.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21, sample_begin=1, sample_stride=2))
            ms.close()
            mc.close()
    ds.close()
    with pytest.raises(rtnw.RtnwError):
        rtnw.MultiContext([])
    with pytest.raises(rtnw.RtnwError):
        rtnw.MultiContext([0, 99])


def test_camera_get_ray_entry_point(rtnw, ctx):
    """rtnw_camera_get_rays = camera::get_ray(s, t) (PSC/camera.h:41-47): exact with a pinhole, inside the lens otherwise"""
    rng = np.random.default_rng(2)
    st = rng.random((4096, 2)).astype(np.float32)
    for aperture in (0.0, 2.0):
        cam = rtnw.make_camera((13, 2, 3), (0, 0, 0), 20, 2.0, aperture, 10.0, 0.25, 0.75)
        r = rtnw.camera_get_rays(ctx, cam, st, seed=4, key_base=100)
        f = lambda a: np.array(list(a), dtype=np.float32)
        org, llc, hor, ver = f(cam.origin), f(cam.lower_left_corner), f(cam.horizontal), f(cam.vertical)
        target = (llc + st[:, :1] * hor) + st[:, 1:] * ver
        assert np.all((r["time"] >= 0.25) & (r["time"] <= 0.75)) and r["time"].std() > 0.1
        assert np.array_equal(r["key"], 100 + np.arange(len(st), dtype=np.uint32))
        if aperture == 0.0:
            assert np.array_equal(r["origin"], np.broadcast_to(org, r["origin"].shape))
            assert np.array_equal(r["direction"], (target - org) - np.float32(0))
        else:
            off = r["origin"] - org
            assert np.all(np.linalg.norm(off, axis=1) <= 1.0 + 1e-5) and np.linalg.norm(off, axis=1).max() > 0.9
            assert np.allclose(r["origin"] + r["direction"], target, rtol=1e-5, atol=1e-5)


def test_division_by_reciprocal(ctx):
    """The leaf tests of a BVH item divide through the reciprocals the ray carries for aabb::hit (rtnw_device.cuh,
    div_by_recip): 2^30 random cases — scene-like values, rays leaving a face plane, zero / tiny / huge components, NaN,
    infinities, any exponent — must give the bits of the IEEE division, as quotients and as hit_box / hit_sphere results."""
    r = ctx.selftest_recip(1 << 30, seed=20261018)
    assert r["box_mismatch"] == 0 and r["sphere_mismatch"] == 0 and r["quotient_mismatch"] == 0, r
    # the shortcut, and real hits, must actually have been exercised
    assert r["box_shortcut"] > (1 << 28) and r["box_hits"] > (1 << 26) and r["sphere_hits"] > (1 << 24), r
