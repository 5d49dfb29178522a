"""Next-event estimation (RTNW_F_NEXT_EVENT, include/rtnw.h): the estimator's C restatement (tests/nee_oracle.c on
tests/light_oracle.c and oracle/rtnw_oracle.c) against the oracle, an analytic image and the exact mode on the CPU; on the GPU
the render against that restatement sample for sample, the path identity the keyed shadow draws give, the reference's own
drand48 fixtures in distribution, the bit-for-bit no-op cases and the render modes."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from test_statistical_parity import PSNR_FLOOR_DB, _criteria, _load, _psnr

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "peter-shirley-ray-tracing-the-next-week_b200" / "bin" / "rtnw_main"

# Mean per-pixel variance of the flagged render over that of the exact one, measured on the C restatement at 32x32, 16 spp
# over 48 seeds (test_restatement_is_unbiased_and_reduces_variance prints it): cornell_box 0.403, cornell_smoke 0.230,
# final_northstar 0.611.  The bounds add a margin.
VAR_RATIO_MAX = {"cornell_box": 0.55, "cornell_smoke": 0.35, "final_northstar": 0.8}


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    """tests/nee_oracle.c compiled with the oracle's flags (oracle/Makefile), plus -fwrapv for the shadow query's depth word,
    into a temporary directory"""
    so = tmp_path_factory.mktemp("nee_oracle") / "libnee_oracle.so"
    subprocess.run([os.environ.get("CC", "gcc"), "-std=gnu11", "-O2", "-ffp-contract=off", "-fwrapv", "-fPIC", "-Wall", "-Wextra",
                    f"-I{ROOT / 'include'}", f"-I{ROOT / 'oracle'}", f"-I{ROOT / 'tests'}", "-shared", "-o", str(so),
                    str(ROOT / "tests" / "nee_oracle.c"), "-lm"], check=True)
    lib = C.CDLL(str(so))
    lib.nee_oracle_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def oracle_render(rtnw, lib, desc_ptr, cam, params):
    """(sums, number of shadow queries) of the restatement"""
    t = rtnw.device_tables(desc_ptr)
    lights = np.ascontiguousarray(t["lights"], dtype=np.float32)
    leaf = np.ascontiguousarray(t["rec_leaf"][lights[:, 7].view(np.int32)], dtype=np.int32)
    out = np.zeros((params.ny, params.nx, 3), np.float32)
    n = C.c_uint64()
    assert lib.nee_oracle_render(C.cast(desc_ptr, C.c_void_p), lights.ctypes.data, leaf.ctypes.data, len(lights),
                                 C.cast(C.pointer(cam), C.c_void_p), C.cast(C.pointer(params), C.c_void_p), out.ctypes.data,
                                 C.byref(n)) == 0
    return out, n.value


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ------------------------------------------------------------------------------------------------ CPU
def test_restatement_without_the_flag_is_the_oracle(rtnw, oracle):
    """without the flag, with the flag and RTNW_F_EMIT off, and with the flag on a scene with no sampleable light, the restatement
    is rtnw_oracle_render bit for bit and traces no shadow ray"""
    import oracle_port as op
    for name, flags_off, flagged in (("cornell_box", 0, (0,)), ("cornell_box", rtnw.F_EMIT, (0, rtnw.F_NEXT_EVENT)),
                                     ("two_perlin", 0, (0, rtnw.F_NEXT_EVENT))):
        hs = rtnw.HostScene(name)
        nx, ny = 24, 24
        cam = hs.camera(nx, ny)
        p = hs.params(nx=nx, ny=ny, ns=3, seed=5)
        p.flags &= ~flags_off
        want = op.render(rtnw, hs.desc_ptr, cam, p)[0]
        for f in flagged:
            q = hs.params(nx=nx, ny=ny, ns=3, seed=5, flags_extra=f)
            q.flags &= ~flags_off
            got, n = oracle_render(rtnw, oracle, hs.desc_ptr, cam, q)
            assert np.array_equal(bits(got), bits(want)) and n == 0, (name, flags_off, f)
        hs.close()


ALBEDO, EMIT, H = (0.5, 0.6, 0.7), 4.0, 1.0  # the floor y = 0, the light y = H over x in [1, 2], z in [-0.5, 0.5]
LIGHT = (1.0, 2.0, -0.5, 0.5)
CAM_Y, FOOT = 5.0, 0.25  # a pinhole straight above the origin; the image sees the floor over x, z in [-FOOT, FOOT]


def floor_scene(rtnw):
    """a lambertian xz floor under a diffuse_light xz rectangle, in one list item"""
    hs = rtnw.HostScene("two_perlin")  # perlin tables
    d = rtnw.SceneDesc()
    C.memmove(C.byref(d), C.byref(hs.desc), C.sizeof(d))
    tex = (rtnw.Texture * 2)()
    tex[0].c[0], tex[0].c[1], tex[0].c[2] = ALBEDO
    tex[1].c[0] = tex[1].c[1] = tex[1].c[2] = EMIT
    mat = (rtnw.Material * 2)()
    mat[0].kind, mat[0].tex = 0, 0  # RTNW_MAT_LAMBERTIAN
    mat[1].kind, mat[1].tex = 3, 1  # RTNW_MAT_DIFFUSE_LIGHT
    xf = (rtnw.XformOp * 1)()
    prim = (rtnw.Prim * 2)()
    for q, v in enumerate((-4.0, 4.0, -4.0, 4.0, 0.0)):
        prim[0].f[q] = v
    for q, v in enumerate(LIGHT + (H,)):
        prim[1].f[q] = v
    prim[0].kx = prim[1].kx = 3  # RTNW_PRIM_RECT_XZ, no flip, no transform
    prim[0].mat, prim[1].mat = 0, 1
    ids = (C.c_int32 * 2)(0, 1)
    item = (rtnw.Item * 1)()
    item[0].kind, item[0].xform, item[0].first, item[0].count = 0, 0, 0, 2
    d.n_items, d.items, d.n_nodes = 1, item, 0
    d.n_prim_slots, d.prims, d.prim_ids = 2, prim, ids
    d.n_xform_ops, d.xforms = 1, xf
    d.n_materials, d.materials, d.n_textures, d.textures = 2, mat, 2, tex
    cam = rtnw.Camera()
    w = 2 * FOOT / CAM_Y  # image plane one unit below the pinhole
    for q, v in enumerate((0.0, CAM_Y, 0.0)):
        cam.origin[q] = v
    for q, v in enumerate((-w / 2, CAM_Y - 1.0, -w / 2)):
        cam.lower_left_corner[q] = v
    cam.horizontal[0], cam.vertical[2] = w, w
    return d, cam, (hs, tex, mat, xf, prim, ids, item)


def floor_mean():
    """the image's expected mean per channel: ALBEDO EMIT times the mean over the floor footprint of the integral of p_ref over
    the directions that meet the light, (2/pi) H^4 / r^6 over the light's area; Gauss-Legendre in all four dimensions"""
    from scipy.special import roots_legendre
    xg, wg = roots_legendre(24)

    def nodes(a, b):
        return (a + b) / 2 + (b - a) / 2 * xg, (b - a) / 2 * wg
    (fx, wfx), (fz, wfz) = nodes(-FOOT, FOOT), nodes(-FOOT, FOOT)
    (lx, wlx), (lz, wlz) = nodes(*LIGHT[:2]), nodes(*LIGHT[2:])
    X, Z, QX, QZ = np.meshgrid(fx, fz, lx, lz, indexing="ij")
    W = np.einsum("i,j,k,l->ijkl", wfx, wfz, wlx, wlz)
    r2 = (X - QX) ** 2 + H ** 2 + (Z - QZ) ** 2
    e = np.sum(W * (2 / np.pi) * H ** 4 / r2 ** 3) / (2 * FOOT) ** 2
    return np.float64(ALBEDO) * EMIT * e


def test_analytic_floor_under_a_rectangle_light(rtnw, oracle):
    """max_depth 1: the mean of the image is the albedo times the emission times p_ref's mass over the light, computed by
    quadrature; the restatement with and without the flag meets it within 4 sigma over independent seeds"""
    d, cam, keep = floor_scene(rtnw)
    ptr = C.pointer(d)
    assert len(rtnw.device_tables(ptr)["lights"]) == 1
    want = floor_mean()
    nx = ny = 32
    for f in (0, rtnw.F_NEXT_EVENT):
        means = []
        for s in range(16):
            p = rtnw.RenderParams(nx, ny, 0, 32, 1, 1, 0.001, rtnw.FLT_MAX, rtnw.BG_BLACK, rtnw.F_EMIT | rtnw.F_DE_NAN | f, 300 + s,
                                  0, 1, 0, 0)
            img, n = oracle_render(rtnw, oracle, ptr, cam, p)
            assert (n > 0) == (f != 0)
            means.append(img.astype(np.float64).mean(axis=(0, 1)) / 32)
        means = np.array(means)
        se = means.std(0, ddof=1) / np.sqrt(len(means))
        print(f"flags {f}: {means.mean(0)} vs {want} (se {se})")
        assert (np.abs(means.mean(0) - want) <= 4 * se).all(), (f, means.mean(0), want, se)


def global_means_and_variance(rtnw, oracle, hs, nx, ny, ns, seeds, flags):
    cam = hs.camera(nx, ny)
    imgs = np.stack([oracle_render(rtnw, oracle, hs.desc_ptr, cam, hs.params(nx=nx, ny=ny, ns=ns, seed=s, flags_extra=flags))[0] / ns
                     for s in seeds]).astype(np.float64)
    return imgs.mean(axis=(1, 2)), imgs.var(axis=0, ddof=1).mean()


@pytest.mark.parametrize("name", ["cornell_box", "cornell_smoke", "final_northstar"])
def test_restatement_is_unbiased_and_reduces_variance(rtnw, oracle, name):
    """the restatement with the flag against itself without it (rtnw_oracle_render, test above): per-channel global means agree
    within 4 sigma over 48 seeds, and the mean per-pixel variance ratio stays below VAR_RATIO_MAX"""
    hs = rtnw.HostScene(name)
    nx = ny = 32
    seeds = range(100, 148)
    g_f, v_f = global_means_and_variance(rtnw, oracle, hs, nx, ny, 16, seeds, rtnw.F_NEXT_EVENT)
    g_e, v_e = global_means_and_variance(rtnw, oracle, hs, nx, ny, 16, seeds, 0)
    se = np.sqrt(g_f.var(0, ddof=1) / len(g_f) + g_e.var(0, ddof=1) / len(g_e))
    z = np.abs(g_f.mean(0) - g_e.mean(0)) / se
    print(f"{name}: global means {g_f.mean(0)} vs {g_e.mean(0)} (z {z}), per-pixel variance ratio {v_f / v_e:.3f}")
    assert (z <= 4).all(), z
    assert v_f / v_e <= VAR_RATIO_MAX[name], v_f / v_e
    hs.close()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def scenes(rtnw, ctx):
    cache = {}

    def get(name):
        if name not in cache:
            hs = rtnw.HostScene(name)
            cache[name] = (hs, ctx.upload(hs.desc_ptr))
        return cache[name]
    yield get
    for hs, ds in cache.values():
        ds.close()
        hs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,nx,ny,ns", [("cornell_box", 48, 48, 4), ("cornell_smoke", 40, 40, 4), ("simple_light", 64, 32, 6),
                                           ("final_northstar", 48, 48, 2), ("earth", 48, 32, 4)])
def test_render_matches_the_restatement_sample_for_sample(rtnw, scenes, oracle, name, nx, ny, ns):
    """the criterion of test_gpu_parity.py::test_render_matches_reference_sample_for_sample; and in the exact traversal the
    flagged render's closest-hit queries are the plain render's plus the restatement's shadow queries, its paths the same"""
    hs, ds = scenes(name)
    cam = hs.camera(nx, ny)
    p = hs.params(nx=nx, ny=ny, ns=ns, seed=1234, flags_extra=rtnw.F_NEXT_EVENT)
    got, st = ds.render(cam, p)
    want, shadows = oracle_render(rtnw, oracle, hs.desc_ptr, cam, p)
    plain, st0 = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=1234))
    assert not np.array_equal(bits(got), bits(plain))
    close = np.isclose(got, want, rtol=2e-5, atol=1e-6).all(axis=2)
    print(f"{name}: {close.mean():.5f} of pixels agree, {shadows} shadow queries for {st.paths} paths")
    assert close.mean() >= 0.99, f"{name}: only {close.mean():.4f} of pixels agree"
    assert abs(got.sum() - want.sum()) <= 2e-3 * abs(want.sum()) + 1e-3
    assert shadows > 0 and st.rays == st0.rays + shadows and st.paths == st0.paths


@pytest.mark.gpu
def test_aovs_are_the_plain_aovs(rtnw, scenes):
    hs, ds = scenes("final_northstar")
    cam = hs.camera(64, 48)
    plain = ds.render_aov(cam, hs.params(nx=64, ny=48, ns=3, seed=8))
    flagged = ds.render_aov(cam, hs.params(nx=64, ny=48, ns=3, seed=8, flags_extra=rtnw.F_NEXT_EVENT))
    for k, v in plain.items():
        assert np.array_equal(bits(flagged[k]), bits(v)), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "cornell_smoke", "final_northstar"])
def test_image_statistics_match_reference_drand48(rtnw, scenes, name):
    """test_statistical_parity.py's three criteria for the flagged render (mean within 0.5 %, 99 % of pixel channels within
    4 sigma, the PSNR floors), and its per-pixel variance against the reference's.  final_northstar meets the mean and PSNR
    criteria (0.025 % off, 30.85 dB against 28.35 dB reference vs reference, one B200) but has 97.38 % of its pixel channels
    within 4 sigma, so its bound is 97 %: 2.57 % lie above the reference's mean and 0.05 % below.  The 4-sigma test takes its
    sigma from both sides' own batches, and this scene's reference means are heavy-tailed (rare paths that find the light from
    dim pixels): a reference batch set without those paths is low and has a small variance.  The exact mode's noise has the
    same tail and covers it; the flagged render's has 0.57 of the variance and does not.  Against the exact mode itself, with
    64 batches on each side, the flagged render holds 99 % (test_pixels_match_the_exact_mode)."""
    g, K, (m_ref, v_ref), (m_b, _) = _load(name)
    nx, ny, spp = int(g["nx"]), int(g["ny"]), int(g["spp"])
    hs, ds = scenes(name)
    cam = hs.camera(nx, ny)
    gpu = np.stack([ds.render(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=900 + k, flags_extra=rtnw.F_NEXT_EVENT))[0] / spp
                    for k in range(K)]).astype(np.float64)
    rel, frac, psnr = _criteria(gpu.mean(0), gpu.var(0, ddof=1) / K, m_ref, v_ref)
    floor = _psnr(m_b, m_ref)
    ratio = gpu.var(0, ddof=1).mean() / g["var_a"].astype(np.float64).mean()
    print(f"{name}: global mean off by {100 * rel:.3f} %, {100 * frac:.3f} % within 4 sigma, PSNR {psnr:.2f} dB "
          f"(reference vs reference {floor:.2f} dB), per-pixel variance ratio {ratio:.3f}")
    assert rel <= 0.005 and frac >= (0.97 if name == "final_northstar" else 0.99)
    assert psnr >= floor - 1.0 and psnr >= PSNR_FLOOR_DB[name]


@pytest.mark.gpu
def test_pixels_match_the_exact_mode(rtnw, scenes):
    """final_northstar at the fixture's size and spp, 64 seeds in each mode: >= 99 % of pixel channels of the flagged mean lie
    within 4 sigma of the exact mode's (99.913 % measured on one B200, every miss above)"""
    g = np.load(ROOT / "tests" / "golden" / "stat_final_northstar.npz")
    nx, ny, spp = int(g["nx"]), int(g["ny"]), int(g["spp"])
    hs, ds = scenes("final_northstar")
    cam = hs.camera(nx, ny)

    def batches(flags, base):
        return np.stack([ds.render(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=base + k, flags_extra=flags))[0] / spp
                         for k in range(64)]).astype(np.float64)
    a, b = batches(rtnw.F_NEXT_EVENT, 900), batches(0, 5000)
    se = np.sqrt(a.var(0, ddof=1) / len(a) + b.var(0, ddof=1) / len(b))
    ok = se > 0
    z = np.abs(a.mean(0) - b.mean(0))[ok] / se[ok]
    print(f"final_northstar: {100 * (z <= 4).mean():.3f} % of pixel channels within 4 sigma of the exact mode")
    assert (z <= 4).mean() >= 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ch01_random", "two_perlin", "two_spheres", "cornell_box"])
def test_no_light_or_no_emission_is_a_bitwise_no_op(rtnw, scenes, name):
    hs, ds = scenes(name)
    cam = hs.camera(40, 30)
    p = hs.params(nx=40, ny=30, ns=4, seed=3)
    if name == "cornell_box":
        p.flags &= ~rtnw.F_EMIT
    a, sa = ds.render(cam, p)
    p.flags |= rtnw.F_NEXT_EVENT
    b, sb = ds.render(cam, p)
    assert np.array_equal(bits(a), bits(b)) and sa.rays == sb.rays


@pytest.mark.gpu
def test_light_sampling_and_next_event_exclude_each_other(rtnw, ctx, scenes):
    hs, ds = scenes("cornell_box")
    cam = hs.camera(32, 32)
    good = hs.params(nx=32, ny=32, ns=2, seed=4, flags_extra=rtnw.F_NEXT_EVENT)
    want, _ = ds.render(cam, good)
    bad = hs.params(nx=32, ny=32, ns=2, seed=4, flags_extra=rtnw.F_NEXT_EVENT | rtnw.F_LIGHT_SAMPLING)
    with pytest.raises(rtnw.RtnwError) as e:
        ds.render(cam, bad)
    assert e.value.code == rtnw.RTNW_ERR_INVALID
    import torch
    buf = torch.zeros((32, 32, 3), dtype=torch.float32, device="cuda")
    with pytest.raises(rtnw.RtnwError) as e:
        ds.render_device(cam, bad, buf.data_ptr())
    assert e.value.code == rtnw.RTNW_ERR_INVALID
    mc = rtnw.MultiContext([0, 0])
    ms = mc.upload(hs.desc_ptr)
    for call in (ms.render, ms.render_aov):
        with pytest.raises(rtnw.RtnwError) as e:
            call(cam, bad)
        assert e.value.code == rtnw.RTNW_ERR_INVALID
    ms.close()
    mc.close()
    again, _ = ds.render(cam, good)
    assert np.array_equal(bits(again), bits(want))


@pytest.mark.gpu
def test_modes(rtnw, ctx, scenes):
    """determinism, the fast traversal, ROTATE shares, rtnw_render_device, an accumulated pixel subset, one sample range,
    DE_NAN off, and rtnw_render_multi / rtnw_render_aov_multi"""
    import torch
    hs, ds = scenes("final_northstar")
    nx, ny, ns = 96, 64, 6
    cam = hs.camera(nx, ny)
    F = rtnw.F_NEXT_EVENT
    p = hs.params(nx=nx, ny=ny, ns=ns, seed=21, flags_extra=F)
    one, st = ds.render(cam, p)
    again, _ = ds.render(cam, p)
    assert np.array_equal(bits(one), bits(again)) and st.paths == nx * ny * ns
    fast, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21, flags_extra=F | rtnw.F_FAST_BVH))
    assert np.isclose(fast, one, rtol=1e-5, atol=1e-6).all(axis=2).mean() > 0.97
    for G in (2, 3):
        parts = sum(ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21, sample_begin=g, sample_stride=G,
                                             flags_extra=F | rtnw.F_ROTATE_SAMPLES))[0] for g in range(G))
        assert np.allclose(parts, one, rtol=1e-5, atol=1e-6), G
    buf = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
    ds.render_device(cam, p, buf.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bits(buf.cpu().numpy()), bits(one))
    begin, stride, count = 5, 7, 600
    pre = np.full((ny, nx, 3), 2.0, np.float32)
    buf = torch.from_numpy(pre.copy()).cuda()
    ds.render_device(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21, flags_extra=F | rtnw.F_ACCUMULATE, pixel_begin=begin,
                                    pixel_stride=stride, pixel_count=count), buf.data_ptr())
    torch.cuda.synchronize()
    got = buf.cpu().numpy().reshape(-1, 3)
    sub = begin + stride * np.arange(count)
    rest = np.setdiff1d(np.arange(nx * ny), sub)
    assert np.allclose(got[sub], 2.0 + one.reshape(-1, 3)[sub], rtol=1e-5, atol=1e-5)
    assert np.array_equal(got[rest], pre.reshape(-1, 3)[rest])
    single, _ = ds.render(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21, flags_extra=F, sample_ranges=1))
    assert np.allclose(single, one, rtol=1e-5, atol=1e-6)
    q = hs.params(nx=nx, ny=ny, ns=ns, seed=21, flags_extra=F)
    q.flags &= ~rtnw.F_DE_NAN
    raw, _ = ds.render(cam, q)
    assert np.isclose(raw, one, rtol=1e-5, atol=1e-6).all(axis=2).mean() > 0.999
    plain_aov = ds.render_aov(cam, hs.params(nx=nx, ny=ny, ns=ns, seed=21))
    for devs in ([0, 0], [0, 0, 0]):
        mc = rtnw.MultiContext(devs)
        ms = mc.upload(hs.desc_ptr)
        a, _ = ms.render(cam, p)
        assert np.allclose(a, one, rtol=1e-5, atol=1e-6), devs
        sums, aov, _, _ = ms.render_aov(cam, p)
        assert np.array_equal(bits(sums), bits(a))
        for k in ("hits", "prim_id"):
            assert np.array_equal(aov[k], plain_aov[k])
        ms.close()
        mc.close()


@pytest.mark.gpu
def test_driver_renders_with_next_event(rtnw, scenes, tmp_path):
    nx, ny, ns = 32, 32, 4
    r = subprocess.run([str(BIN), "cornell_box", str(nx), str(ny), str(ns), str(tmp_path / "out.ppm"), "--nee"], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    hs, ds = scenes("cornell_box")
    sums, _ = ds.render(hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=1, flags_extra=rtnw.F_NEXT_EVENT))
    rtnw.write_ppm(str(tmp_path / "want.ppm"), sums, ns)
    assert (tmp_path / "out.ppm").read_bytes() == (tmp_path / "want.ppm").read_bytes()
