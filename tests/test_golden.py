"""Golden fixtures (tests/golden/*.npz, generated from the reference itself by tests/golden/make_golden.py):
  * CPU: the C restatement of the oracle reproduces every fixture bit for bit (no reference needed at run time);
  * GPU: the CUDA path, through the C-ABI, reproduces ids / t / p / normal bit for bit, uv within 1e-5, and the
    sample-for-sample renders within the tolerance of test_gpu_parity.py."""
from pathlib import Path

import numpy as np
import pytest

import oracle_port as op
from raysets import FLT_MAX, assert_hits_equal, scene_with_material

GOLD = Path(__file__).resolve().parent / "golden"
TRACE = sorted(p.stem[len("trace_"):] for p in GOLD.glob("trace_*.npz"))
RENDER = sorted(p.stem[len("render_"):] for p in GOLD.glob("render_*.npz"))


def scene_name(stem):
    return stem[:-4] + "+bvh" if stem.endswith("_bvh") else stem


def test_fixtures_are_present():
    assert len(TRACE) >= 10 and len(RENDER) >= 9 and (GOLD / "units.npz").exists()


@pytest.mark.parametrize("stem", TRACE)
def test_oracle_port_reproduces_golden_hits(rtnw, stem):
    g = np.load(GOLD / f"trace_{stem}.npz")
    hs = rtnw.HostScene(scene_name(stem))
    seed = int(g["seed"])
    assert_hits_equal(op.trace(rtnw, hs.desc_ptr, g["rays"], 0.001, FLT_MAX, seed=seed), g["hits_a"], uv_tol=0)
    assert_hits_equal(op.trace(rtnw, hs.desc_ptr, g["rays"], 0.0, 400.0, seed=seed), g["hits_b"], uv_tol=0)


@pytest.mark.parametrize("stem", RENDER)
def test_oracle_port_reproduces_golden_renders(rtnw, stem):
    g = np.load(GOLD / f"render_{stem}.npz")
    hs = rtnw.HostScene(scene_name(stem))
    nx, ny, ns = int(g["nx"]), int(g["ny"]), int(g["ns"])
    got, st = op.render(rtnw, hs.desc_ptr, hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=int(g["seed"])))
    assert np.array_equal(got.view(np.uint32), g["sums"].view(np.uint32))
    assert st["rays"] == float(g["rays"])


def test_oracle_port_reproduces_golden_units(rtnw):
    g = np.load(GOLD / "units.npz")
    hs = rtnw.HostScene("two_perlin")
    d = hs.desc
    kinds = [d.textures[i].kind for i in range(d.n_textures)]
    assert np.array_equal(op.eval_perlin(rtnw, hs.desc_ptr, 0, g["xyz"]), g["noise"])
    assert np.array_equal(op.eval_perlin(rtnw, hs.desc_ptr, 1, g["xyz"]), g["turb"])
    assert np.array_equal(op.eval_texture(rtnw, hs.desc_ptr, kinds.index(1), g["uvp"]), g["checker"])
    assert np.array_equal(op.eval_texture(rtnw, hs.desc_ptr, kinds.index(2), g["uvp"]), g["noise_tex"])
    he = rtnw.HostScene("earth")
    ke = [he.desc.textures[i].kind for i in range(he.desc.n_textures)]
    assert np.array_equal(op.eval_texture(rtnw, he.desc_ptr, ke.index(3), g["uvp"]), g["image"])
    cam = rtnw.HostScene("ch01_random").camera(200, 100)
    got = op.camera_rays(rtnw, cam, 200, 100, g["cam_ij"], g["cam_sample"], seed=77)
    for f in ("origin", "direction", "time", "key"):
        assert np.array_equal(got[f], g["cam_rays"][f]), f


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("stem", TRACE)
def test_cuda_reproduces_golden_hits(rtnw, ctx, stem):
    g = np.load(GOLD / f"trace_{stem}.npz")
    hs = rtnw.HostScene(scene_name(stem))
    ds = ctx.upload(hs.desc_ptr)
    seed = int(g["seed"])
    assert_hits_equal(ds.trace(g["rays"], 0.001, FLT_MAX, seed=seed), g["hits_a"])
    assert_hits_equal(ds.trace(g["rays"], 0.0, 400.0, seed=seed), g["hits_b"])
    ds.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stem", RENDER)
def test_cuda_reproduces_golden_renders(rtnw, ctx, stem):
    g = np.load(GOLD / f"render_{stem}.npz")
    hs = rtnw.HostScene(scene_name(stem))
    ds = ctx.upload(hs.desc_ptr)
    nx, ny, ns = int(g["nx"]), int(g["ny"]), int(g["ns"])
    got, st = ds.render(hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=int(g["seed"])))
    close = np.isclose(got, g["sums"], rtol=2e-5, atol=1e-6).all(axis=2)
    assert close.mean() >= 0.99, f"{stem}: only {close.mean():.4f} of pixels agree with the reference"
    assert abs(st.rays - float(g["rays"])) <= 0.003 * float(g["rays"])
    ds.close()


@pytest.mark.gpu
def test_cuda_reproduces_golden_units(rtnw, ctx):
    g = np.load(GOLD / "units.npz")
    hs = rtnw.HostScene("two_perlin")
    ds = ctx.upload(hs.desc_ptr)
    d = hs.desc
    kinds = [d.textures[i].kind for i in range(d.n_textures)]
    assert np.array_equal(ds.eval_perlin(0, g["xyz"]), g["noise"])
    assert np.array_equal(ds.eval_perlin(1, g["xyz"]), g["turb"])
    assert (np.all(ds.eval_texture(kinds.index(1), g["uvp"]) == g["checker"], axis=1)).mean() > 0.998
    assert np.allclose(ds.eval_texture(kinds.index(2), g["uvp"]), g["noise_tex"], rtol=0, atol=2e-6)
    ds.close()
    he = rtnw.HostScene("earth")
    de = ctx.upload(he.desc_ptr)
    ke = [he.desc.textures[i].kind for i in range(he.desc.n_textures)]
    assert np.array_equal(de.eval_texture(ke.index(3), g["uvp"]), g["image"])
    de.close()
    cam = rtnw.HostScene("ch01_random").camera(200, 100)
    got = rtnw.camera_rays(ctx, cam, 200, 100, g["cam_ij"], g["cam_sample"], seed=77)
    for f in ("origin", "direction", "time", "key"):
        assert np.array_equal(got[f], g["cam_rays"][f]), f


SCATTER_MATERIALS = ["lambertian", "metal", "dielectric", "light", "isotropic"]


def _golden_scatter_scene(rtnw, g, name):
    """a one-sphere scene whose material 0 is the fixture's row {kind, tex_kind, r, g, b, fuzz_or_ri, scale, 0}"""
    row = g[f"{name}_row"]
    return scene_with_material(rtnw, int(row[0]), tuple(float(x) for x in row[2:5]), float(row[5]), float(row[6]))


@pytest.mark.parametrize("name", SCATTER_MATERIALS)
def test_oracle_port_reproduces_golden_scatter(rtnw, name):
    g = np.load(GOLD / "units.npz")
    d, keep = _golden_scatter_scene(rtnw, g, name)
    sc, att, em, flag = op.scatter(rtnw, d, g["sc_rays"], g["sc_hits"], seed=31)
    for f in ("origin", "direction", "time"):
        assert np.array_equal(sc[f], g[f"{name}_sc"][f], equal_nan=True), f
    assert np.array_equal(att, g[f"{name}_att"]) and np.array_equal(em, g[f"{name}_em"]) and np.array_equal(flag, g[f"{name}_flag"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCATTER_MATERIALS)
def test_cuda_reproduces_golden_scatter(rtnw, ctx, name):
    """scatter() / emitted() on the GPU against the reference's values on the same stream (units.npz), with the rules of
    test_gpu_parity.py::test_scatter_and_emitted_same_stream"""
    g = np.load(GOLD / "units.npz")
    d, keep = _golden_scatter_scene(rtnw, g, name)
    ds = ctx.upload(d)
    sc, att, em, flag = ds.scatter(g["sc_rays"], g["sc_hits"], seed=31)
    ds.close()
    assert np.array_equal(flag, g[f"{name}_flag"]) and np.array_equal(em, g[f"{name}_em"]) and np.array_equal(att, g[f"{name}_att"])
    for f in ("origin", "time"):
        assert np.array_equal(sc[f], g[f"{name}_sc"][f]), f
    a, b = sc["direction"], g[f"{name}_sc"]["direction"]
    same = np.all((a == b) | (np.isnan(a) & np.isnan(b)), axis=1)
    # dielectric: schlick() goes through pow() in double on the CPU, so a draw within an ulp of reflect_prob may flip
    assert (~same).sum() <= (1 if name == "dielectric" else 0)


def _epilogue_cases():
    g = np.load(GOLD / "epilogue.npz")
    for ns in (1, 7, 10, 100, 1000):
        yield ns, g[f"sums_{ns}"], g[f"clamped_{ns}"], g[f"raw_{ns}"]


def test_host_epilogue_reproduces_the_references_own_lines(rtnw):
    """rtnw_host_quantize against PSC/main.cpp:315-325 as compiled from the reference's own text (ref_epilogue in the
    harness, committed as tests/golden/epilogue.npz): quantisation boundaries +-1 ulp, lights > 1, zero, huge, five ns"""
    for ns, sums, clamped, raw in _epilogue_cases():
        assert np.array_equal(rtnw.quantize(sums, ns, clamp255=True), clamped), ns
        assert np.array_equal(rtnw.quantize(sums, ns, clamp255=False), raw), ns


def test_epilogue_fixture_matches_the_live_reference():
    import ref_oracle as ro
    if not ro.available():
        pytest.skip("compiled reference not present")
    for ns, sums, clamped, raw in _epilogue_cases():
        assert np.array_equal(ro.epilogue(sums, ns, True), clamped) and np.array_equal(ro.epilogue(sums, ns, False), raw)


@pytest.mark.gpu
def test_device_epilogue_reproduces_the_references_own_lines(rtnw, ctx):
    """k_quantize (rtnw_quantize_device) bit for bit against the same fixture"""
    import torch
    for ns, sums, clamped, raw in _epilogue_cases():
        ny, nx, _ = sums.shape
        dev = torch.from_numpy(sums).cuda()
        assert np.array_equal(ctx.quantize_device(dev.data_ptr(), nx, ny, ns, clamp255=True), clamped), ns
        assert np.array_equal(ctx.quantize_device(dev.data_ptr(), nx, ny, ns, clamp255=False), raw), ns


def _bilinear_numpy(img, u, v):
    """numpy float32 restatement of the bilinear option (texel centres at i + 0.5, flipped u and v, edges clamped)"""
    ny, nx, _ = img.shape
    f = np.float32
    fx = (f(1) - u) * f(nx) - f(0.5)
    fy = (f(1) - v) * f(ny) - f(0.5)
    x0, y0 = np.floor(fx), np.floor(fy)
    wx, wy = (fx - x0)[:, None], (fy - y0)[:, None]
    i0, i1 = np.clip(x0.astype(np.int64), 0, nx - 1), np.clip(x0.astype(np.int64) + 1, 0, nx - 1)
    j0, j1 = np.clip(y0.astype(np.int64), 0, ny - 1), np.clip(y0.astype(np.int64) + 1, 0, ny - 1)
    c = lambda j, i: img[j, i].astype(np.float32) / f(255.0)
    top = (f(1) - wx) * c(j0, i0) + wx * c(j0, i1)
    bot = (f(1) - wx) * c(j1, i0) + wx * c(j1, i1)
    return (f(1) - wy) * top + wy * bot


def _bilinear_case(rtnw):
    import ctypes as C
    hs = rtnw.HostScene("earth_bilinear")
    d = hs.desc
    tex = [i for i in range(d.n_textures) if d.textures[i].kind == 3][0]
    t = d.textures[tex]
    assert t.flags & rtnw.TEXF_BILINEAR
    img = np.frombuffer(C.string_at(C.addressof(d.images.contents) + t.i0, 3 * t.i1 * t.i2), dtype=np.uint8).reshape(t.i2, t.i1, 3)
    rng = np.random.default_rng(8)
    uv = np.concatenate([rng.random((4000, 2)), [[0, 0], [1, 1], [0, 1], [1, 0], [0.5, 0.5]], rng.random((200, 2)) * 1e-3,
                         1 - rng.random((200, 2)) * 1e-3]).astype(np.float32)
    uvp = np.concatenate([uv, np.zeros((len(uv), 3), np.float32)], axis=1)
    return hs, tex, img, uv, uvp


def test_bilinear_image_texture_option_oracle(rtnw):
    """image_texture's bilinear option (SURVEY §8 f3; not in the reference): the C restatement against a numpy restatement,
    and the nearest-texel default untouched by the flag's existence"""
    hs, tex, img, uv, uvp = _bilinear_case(rtnw)
    got = op.eval_texture(rtnw, hs.desc_ptr, tex, uvp)
    assert np.allclose(got, _bilinear_numpy(img, uv[:, 0], uv[:, 1]), rtol=0, atol=2e-7)
    near = rtnw.HostScene("earth")
    tn = [i for i in range(near.desc.n_textures) if near.desc.textures[i].kind == 3][0]
    assert near.desc.textures[tn].flags == 0
    assert not np.allclose(op.eval_texture(rtnw, near.desc_ptr, tn, uvp), got, atol=1e-3)


@pytest.mark.gpu
def test_bilinear_image_texture_option_gpu(rtnw, ctx):
    hs, tex, img, uv, uvp = _bilinear_case(rtnw)
    ds = ctx.upload(hs.desc_ptr)
    got = ds.eval_texture(tex, uvp)
    assert np.allclose(got, _bilinear_numpy(img, uv[:, 0], uv[:, 1]), rtol=0, atol=2e-7)
    assert np.array_equal(got, op.eval_texture(rtnw, hs.desc_ptr, tex, uvp))
    a, _ = ds.render(hs.camera(48, 48), hs.params(nx=48, ny=48, ns=4, seed=3))
    b, _ = op.render(rtnw, hs.desc_ptr, hs.camera(48, 48), hs.params(nx=48, ny=48, ns=4, seed=3))
    assert np.isclose(a, b, rtol=2e-5, atol=1e-6).all(axis=2).mean() > 0.99
    ds.close()


def _readme_noise_textures(rtnw):
    """{1,2,3} -> (HostScene, texture index) of the Chapter 4 noise drafts (README.md:516-630)"""
    out = {}
    for v in (1, 2, 3):
        hs = rtnw.HostScene(f"perlin_v{v}")
        tex = [i for i in range(hs.desc.n_textures) if hs.desc.textures[i].kind == 3 + v]
        assert len(tex) == 1
        out[v] = (hs, tex[0])
    return out


def test_oracle_port_reproduces_readme_noise_units(rtnw):
    g = np.load(GOLD / "units_readme_noise.npz")
    for v, (hs, tex) in _readme_noise_textures(rtnw).items():
        assert np.array_equal(op.eval_texture(rtnw, hs.desc_ptr, tex, g["uvp"]), g[f"v{v}"]), v


@pytest.mark.gpu
def test_cuda_reproduces_readme_noise_units(rtnw, ctx):
    """the Chapter 4 noise drafts on the GPU: bit for bit against the harness-side restatement's values"""
    g = np.load(GOLD / "units_readme_noise.npz")
    for v, (hs, tex) in _readme_noise_textures(rtnw).items():
        ds = ctx.upload(hs.desc_ptr)
        assert np.array_equal(ds.eval_texture(tex, g["uvp"]), g[f"v{v}"]), v
        ds.close()
