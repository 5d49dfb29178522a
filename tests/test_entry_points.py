"""The query entry points of include/rtnw.h through the raw C-ABI: empty input, rejected arguments, and that a batch gives
the same bits as the same elements split over two calls.  Each call stages its inputs and outputs in one device
allocation, so a span laid out at a wrong offset or over another span shows up as a batch that differs from its halves."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SCENE = "two_perlin"  # a checker texture with its two children, a noise texture and the perlin tables
NX, NY = 64, 48


@pytest.fixture(scope="module")
def scene(rtnw, ctx):
    hs = rtnw.HostScene(SCENE)
    ds = ctx.upload(hs.desc_ptr)
    yield hs, ds
    ds.close()
    hs.close()


def _lib(rtnw):
    return rtnw.device_lib()


def _camera_rays(rtnw, ctx, hs, n, seed=5):
    rng = np.random.default_rng(n)
    ij = np.stack([rng.integers(0, NX, n), rng.integers(0, NY, n)], axis=1).astype(np.int32)
    sample = rng.integers(0, 100, n).astype(np.int32)
    return ij, sample, rtnw.camera_rays(ctx, hs.camera(NX, NY), NX, NY, ij, sample, seed=seed)


def _inputs(rtnw, ctx, hs, n):
    rng = np.random.default_rng(1000 + n)
    xyz = rng.normal(scale=3, size=(n, 3)).astype(np.float32)
    uvp = np.concatenate([rng.random((n, 2)).astype(np.float32), xyz], axis=1)
    st = rng.random((n, 2)).astype(np.float32)
    ij, sample, rays = _camera_rays(rtnw, ctx, hs, n)
    return dict(xyz=xyz, uvp=uvp, st=st, ij=ij, sample=sample, rays=rays)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8).tobytes()


def test_empty_input_returns_ok(rtnw, ctx, scene):
    hs, ds = scene
    L = _lib(rtnw)
    cam = hs.camera(NX, NY)
    assert L.rtnw_trace(ctx._h, ds._h, None, 0, 0.001, 1e30, 0, 1, None) == rtnw.RTNW_OK
    assert L.rtnw_trace(ctx._h, ds._h, None, 0, 0.001, 1e30, rtnw.F_FAST_BVH, 1, None) == rtnw.RTNW_OK
    assert L.rtnw_eval_texture(ctx._h, ds._h, 0, None, 0, None) == rtnw.RTNW_OK
    for which in (0, 1):
        assert L.rtnw_eval_perlin(ctx._h, ds._h, which, None, 0, None) == rtnw.RTNW_OK
    assert L.rtnw_scatter(ctx._h, ds._h, None, None, 0, 1, None, None, None, None) == rtnw.RTNW_OK
    assert L.rtnw_camera_rays(ctx._h, C.byref(cam), NX, NY, None, None, 0, 1, None) == rtnw.RTNW_OK
    assert L.rtnw_camera_get_rays(ctx._h, C.byref(cam), None, 0, 1, 0, None) == rtnw.RTNW_OK


def _valid_results(rtnw, ctx, hs, ds, dev_sums):
    """one valid call of every entry point the rejection test exercises, as bytes"""
    inp = _inputs(rtnw, ctx, hs, 37)
    cam = hs.camera(NX, NY)
    hits = ds.trace(inp["rays"], seed=3)
    hit = hits["prim_id"] >= 0  # scatter takes hits only: a miss has no material
    sc = ds.scatter(inp["rays"][hit], hits[hit], seed=3)
    return [_bits(hits), _bits(ds.trace(inp["rays"], flags=rtnw.F_FAST_BVH, seed=3)), _bits(ds.eval_texture(0, inp["uvp"])),
            _bits(ds.eval_perlin(1, inp["xyz"])), b"".join(_bits(x) for x in sc),
            _bits(rtnw.camera_rays(ctx, cam, NX, NY, inp["ij"], inp["sample"], seed=7)),
            _bits(rtnw.camera_get_rays(ctx, cam, inp["st"], seed=7, key_base=11)),
            _bits(ctx.quantize_device(dev_sums.data_ptr(), NX, NY, 4))]


def test_rejected_arguments_leave_the_context_usable(rtnw, ctx, scene):
    import torch
    hs, ds = scene
    L = _lib(rtnw)
    cam = hs.camera(NX, NY)
    n = 8
    inp = _inputs(rtnw, ctx, hs, n)
    rays, uvp, xyz, st, ij, sample = inp["rays"], inp["uvp"], inp["xyz"], inp["st"], inp["ij"], inp["sample"]
    hits = ds.trace(rays, seed=3)
    rays_h, hits_h = rays[hits["prim_id"] >= 0], hits[hits["prim_id"] >= 0]
    n_h = len(hits_h)
    assert n_h > 0
    hit_out = np.zeros(n, dtype=rtnw.HIT_DTYPE)
    ray_out = np.zeros(n, dtype=rtnw.RAY_DTYPE)
    f3 = np.zeros((n, 3), np.float32)
    f1 = np.zeros(n, np.float32)
    i1 = np.zeros(n, np.int32)
    q_out = np.zeros((NY, NX, 3), np.int32)
    sums = torch.rand((NY, NX, 3), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(9)) * 4
    before = _valid_results(rtnw, ctx, hs, ds, sums)

    def bad_hits(mat_id):
        h = hits_h.copy()
        h["mat_id"][n_h // 2] = mat_id
        return h.ctypes.data, h  # keep the copy alive with the pointer

    n_tex, n_mat = hs.desc.n_textures, hs.desc.n_materials
    h_neg, keep_neg = bad_hits(-1)
    h_big, keep_big = bad_hits(n_mat)
    p = lambda a: a.ctypes.data  # noqa: E731
    calls = {
        "trace: null scene": lambda: L.rtnw_trace(ctx._h, None, p(rays), n, 0.001, 1e30, 0, 1, p(hit_out)),
        "trace: null rays": lambda: L.rtnw_trace(ctx._h, ds._h, None, n, 0.001, 1e30, 0, 1, p(hit_out)),
        "trace: null out": lambda: L.rtnw_trace(ctx._h, ds._h, p(rays), n, 0.001, 1e30, rtnw.F_FAST_BVH, 1, None),
        "texture: tex_id -1": lambda: L.rtnw_eval_texture(ctx._h, ds._h, -1, p(uvp), n, p(f3)),
        "texture: tex_id n_textures": lambda: L.rtnw_eval_texture(ctx._h, ds._h, n_tex, p(uvp), n, p(f3)),
        "texture: null uvp": lambda: L.rtnw_eval_texture(ctx._h, ds._h, 0, None, n, p(f3)),
        "texture: null scene": lambda: L.rtnw_eval_texture(ctx._h, None, 0, p(uvp), n, p(f3)),
        "perlin: which 2": lambda: L.rtnw_eval_perlin(ctx._h, ds._h, 2, p(xyz), n, p(f1)),
        "perlin: which -1": lambda: L.rtnw_eval_perlin(ctx._h, ds._h, -1, p(xyz), n, p(f1)),
        "perlin: null out": lambda: L.rtnw_eval_perlin(ctx._h, ds._h, 0, p(xyz), n, None),
        "scatter: mat_id -1": lambda: L.rtnw_scatter(ctx._h, ds._h, p(rays_h), h_neg, n_h, 1, p(ray_out), p(f3), p(f3), p(i1)),
        "scatter: mat_id n_materials": lambda: L.rtnw_scatter(ctx._h, ds._h, p(rays_h), h_big, n_h, 1, p(ray_out), p(f3), p(f3), p(i1)),
        "scatter: null flag": lambda: L.rtnw_scatter(ctx._h, ds._h, p(rays_h), p(hits_h), n_h, 1, p(ray_out), p(f3), p(f3), None),
        "camera_rays: nx 0": lambda: L.rtnw_camera_rays(ctx._h, C.byref(cam), 0, NY, p(ij), p(sample), n, 1, p(ray_out)),
        "camera_rays: ny -1": lambda: L.rtnw_camera_rays(ctx._h, C.byref(cam), NX, -1, p(ij), p(sample), n, 1, p(ray_out)),
        "camera_rays: nx 0, n 0": lambda: L.rtnw_camera_rays(ctx._h, C.byref(cam), 0, NY, None, None, 0, 1, None),
        "camera_rays: null sample": lambda: L.rtnw_camera_rays(ctx._h, C.byref(cam), NX, NY, p(ij), None, n, 1, p(ray_out)),
        "get_rays: null camera": lambda: L.rtnw_camera_get_rays(ctx._h, None, p(st), n, 1, 0, p(ray_out)),
        "get_rays: null st": lambda: L.rtnw_camera_get_rays(ctx._h, C.byref(cam), None, n, 1, 0, p(ray_out)),
        "quantize: ns 0": lambda: L.rtnw_quantize_device(ctx._h, C.c_void_p(sums.data_ptr()), NX, NY, 0, 1, p(q_out)),
        "quantize: ns -1": lambda: L.rtnw_quantize_device(ctx._h, C.c_void_p(sums.data_ptr()), NX, NY, -1, 1, p(q_out)),
        "quantize: nx 0": lambda: L.rtnw_quantize_device(ctx._h, C.c_void_p(sums.data_ptr()), 0, NY, 4, 1, p(q_out)),
        "quantize: null input": lambda: L.rtnw_quantize_device(ctx._h, None, NX, NY, 4, 1, p(q_out)),
        "quantize: null output": lambda: L.rtnw_quantize_device(ctx._h, C.c_void_p(sums.data_ptr()), NX, NY, 4, 1, None),
        "selftest: null out": lambda: L.rtnw_selftest_recip(ctx._h, 16, 1, None),
        "fp32 peak: null out": lambda: L.rtnw_measure_fp32_peak(ctx._h, None),
    }
    for what, call in calls.items():
        assert call() == rtnw.RTNW_ERR_INVALID, what
    del keep_neg, keep_big
    assert _valid_results(rtnw, ctx, hs, ds, sums) == before


@pytest.mark.parametrize("n", [1, 3, 37, 1000])
def test_batch_equals_split(rtnw, ctx, scene, n):
    hs, ds = scene
    cam = hs.camera(NX, NY)
    inp = _inputs(rtnw, ctx, hs, n)
    k = max(1, n // 3)  # uneven halves; n = 1 splits into one element and an empty call

    def split(f, *arrays):
        whole = f(*arrays)
        parts = [f(*(a[:k] for a in arrays)), f(*(a[k:] for a in arrays))]
        assert _bits(whole) == _bits(np.concatenate(parts)), f"n={n} split at {k}"

    for flags in (0, rtnw.F_FAST_BVH):
        split(lambda r: ds.trace(r, flags=flags, seed=3), inp["rays"])
    for tex in range(hs.desc.n_textures):
        split(lambda u: ds.eval_texture(tex, u), inp["uvp"])
    for which in (0, 1):
        split(lambda x: ds.eval_perlin(which, x), inp["xyz"])
    split(lambda ij, s: rtnw.camera_rays(ctx, cam, NX, NY, ij, s, seed=7), inp["ij"], inp["sample"])
    whole = rtnw.camera_get_rays(ctx, cam, inp["st"], seed=7, key_base=100)
    first = rtnw.camera_get_rays(ctx, cam, inp["st"][:k], seed=7, key_base=100)
    second = rtnw.camera_get_rays(ctx, cam, inp["st"][k:], seed=7, key_base=100 + k)
    assert _bits(whole) == _bits(np.concatenate([first, second]))
