"""First-hit feature buffers (rtnw_render_aov, DeviceScene.render_aov, rtnw_main --aov) on the GPU: against their restatement on
the C oracle of the reference (tests/aov_oracle.c on oracle/rtnw_oracle.c) pixel for pixel, against the render's own first closest hit, fast mode,
determinism, argument errors and the driver's PFM files."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from test_pfm import read_pfm

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "peter-shirley-ray-tracing-the-next-week_b200" / "bin" / "rtnw_main"
KEYS = ("albedo", "normal", "depth", "hits", "prim_id")


@pytest.fixture(scope="module")
def scenes(rtnw, ctx):
    """name -> (HostScene, DeviceScene), uploaded once for the module"""
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


@pytest.fixture(scope="module")
def oracle_aov(rtnw, tmp_path_factory):
    """rtnw_oracle_aov of tests/aov_oracle.c, compiled with the oracle's flags (oracle/Makefile) into a temporary directory:
    (desc_ptr, cam, params) -> dict of the five buffers"""
    so = tmp_path_factory.mktemp("aov_oracle") / "libaov_oracle.so"
    subprocess.run([os.environ.get("CC", "gcc"), "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                    f"-I{ROOT / 'include'}", f"-I{ROOT / 'oracle'}", "-shared", "-o", str(so), str(ROOT / "tests" / "aov_oracle.c"), "-lm"],
                   check=True)
    lib = C.CDLL(str(so))
    lib.rtnw_oracle_aov.argtypes = [C.c_void_p] * 8

    def run(desc_ptr, cam, params):
        ny, nx = params.ny, params.nx
        out = dict(albedo=np.zeros((ny, nx, 3), np.float32), normal=np.zeros((ny, nx, 3), np.float32),
                   depth=np.zeros((ny, nx), np.float32), hits=np.zeros((ny, nx), np.int32), prim_id=np.zeros((ny, nx), np.int32))
        rc = lib.rtnw_oracle_aov(C.cast(desc_ptr, C.c_void_p), C.cast(C.pointer(cam), C.c_void_p), C.cast(C.pointer(params), C.c_void_p),
                                 *(out[k].ctypes.data for k in KEYS))
        assert rc == 0
        return out
    return run


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def constant_textures_only(rtnw, hs):
    d = hs.desc
    return all(d.textures[t].kind == 0 for t in range(d.n_textures))  # RTNW_TEX_CONSTANT


def assert_matches_oracle(rtnw, hs, got, want):
    for k in ("hits", "prim_id"):
        assert np.array_equal(got[k], want[k]), f"{k}: {(got[k] != want[k]).sum()} pixels differ"
    for k in ("normal", "depth"):
        same = bits(got[k]) == bits(want[k])
        assert same.all(), f"{k}: {(~same).sum()} values differ"
    if constant_textures_only(rtnw, hs):  # every albedo value is a table constant, the sky, or (1,1,1): exact
        assert np.array_equal(bits(got["albedo"]), bits(want["albedo"]))
    else:  # sinf, perlin and atan2f / asinf u,v are within 2e-6 / 1e-5 of glibc: the project's image bar
        close = np.isclose(got["albedo"], want["albedo"], rtol=2e-5, atol=1e-6).all(axis=2).mean()
        assert close >= 0.99, f"albedo: only {close:.4f} of pixels agree with the oracle"


@pytest.mark.parametrize("name, nx, ny", [("cornell_box", 64, 64), ("cornell_smoke", 64, 64), ("final_northstar", 64, 64),
                                          ("ch01_random", 100, 50), ("two_perlin", 64, 32), ("earth", 64, 32)])
def test_aov_matches_the_oracle_on_every_pixel(rtnw, scenes, oracle_aov, name, nx, ny):
    hs, ds = scenes(name)
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=4, seed=7)
    st = rtnw.Stats()
    got = ds.render_aov(cam, params, st)
    want = oracle_aov(hs.desc_ptr, cam, params)
    assert (got["hits"] > 0).mean() > 0.05  # earth at 64x32: the sphere and the light cover 9 % of the frame
    assert_matches_oracle(rtnw, hs, got, want)
    assert st.paths == st.rays == nx * ny * 4 and st.kernel_launches == 1 and st.kernel_ms > 0


@pytest.mark.parametrize("name", ["final_northstar", "cornell_smoke"])
def test_aov_first_hit_is_the_render_paths_first_hit(rtnw, ctx, scenes, oracle_aov, name):
    nx, ny = 64, 64
    hs, ds = scenes(name)
    cam = hs.camera(nx, ny)
    params = hs.params(nx=nx, ny=ny, ns=1, seed=7)
    got = ds.render_aov(cam, params)
    j, i = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    ij = np.stack([i.ravel(), j.ravel()], axis=1)  # pixel p = j*nx + i in buffer order
    rays = rtnw.camera_rays(ctx, cam, nx, ny, ij, np.zeros(len(ij), np.int32), seed=7)
    hit = ds.trace(rays, params.t_min, rtnw.FLT_MAX, flags=0, seed=7)
    assert np.array_equal(got["prim_id"].ravel(), hit["prim_id"])
    d = rays["direction"]
    length = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    assert np.array_equal(bits(got["depth"]).ravel(), bits(np.where(hit["prim_id"] >= 0, hit["t"] * length, np.float32(0))))
    # sample 7 onwards: the sample index reaches the path stream and the medium key
    later = hs.params(nx=nx, ny=ny, ns=3, seed=7, sample_begin=7)
    assert_matches_oracle(rtnw, hs, ds.render_aov(cam, later), oracle_aov(hs.desc_ptr, cam, later))


@pytest.mark.parametrize("name", ["final_northstar", "final+bvh"])
def test_fast_mode_gives_the_same_hits_and_depth(rtnw, ctx, scenes, name):
    nx, ny = 96, 96
    hs, ds = scenes(name)
    cam = hs.camera(nx, ny)
    exact = ds.render_aov(cam, hs.params(nx=nx, ny=ny, ns=4, seed=3))
    fast = ds.render_aov(cam, hs.params(nx=nx, ny=ny, ns=4, seed=3, flags_extra=rtnw.F_FAST_BVH))
    assert np.array_equal(exact["hits"], fast["hits"])
    assert np.array_equal(bits(exact["depth"]), bits(fast["depth"]))
    other = np.argwhere(exact["prim_id"] != fast["prim_id"])
    assert len(other) < 0.05 * nx * ny
    if len(other):  # a tie: the sample's first ray has another leaf at the same t
        ij = np.stack([other[:, 1], other[:, 0]], axis=1)
        rays = rtnw.camera_rays(ctx, cam, nx, ny, ij, np.zeros(len(ij), np.int32), seed=3)
        a = ds.trace(rays, hs.view.t_min, rtnw.FLT_MAX, flags=0, seed=3)
        b = ds.trace(rays, hs.view.t_min, rtnw.FLT_MAX, flags=rtnw.F_FAST_BVH, seed=3)
        assert np.array_equal(a["prim_id"], exact["prim_id"][other[:, 0], other[:, 1]])
        assert np.array_equal(b["prim_id"], fast["prim_id"][other[:, 0], other[:, 1]])
        assert np.array_equal(bits(a["t"]), bits(b["t"]))


def test_aov_is_deterministic_and_handles_deep_trees(rtnw, scenes):
    hs, ds = scenes("final_northstar")
    cam, params = hs.camera(80, 60), hs.params(nx=80, ny=60, ns=4, seed=9)
    a, b = ds.render_aov(cam, params), ds.render_aov(cam, params)
    for k in KEYS:
        assert a[k].tobytes() == b[k].tobytes(), k
    hs2, ds2 = scenes("stress_shells+bvh")
    out = ds2.render_aov(hs2.camera(64, 48), hs2.params(nx=64, ny=48, ns=2, seed=1))  # raises on a task stack overflow
    assert (out["hits"] > 0).any()


def test_rejected_parameters_leave_the_context_usable(rtnw, scenes):
    hs, ds = scenes("cornell_box")
    cam = hs.camera(32, 32)
    before, _ = ds.render(cam, hs.params(nx=32, ny=32, ns=2, seed=4))
    bad = [hs.params(nx=32, ny=32, ns=2, flags_extra=rtnw.F_ROTATE_SAMPLES), hs.params(nx=32, ny=32, ns=2, flags_extra=rtnw.F_ACCUMULATE),
           hs.params(nx=32, ny=32, ns=2, pixel_count=4), hs.params(nx=32, ny=32, ns=0)]
    for p in bad:
        with pytest.raises(rtnw.RtnwError) as e:
            ds.render_aov(cam, p)
        assert e.value.code == rtnw.RTNW_ERR_INVALID
    ok = hs.params(nx=32, ny=32, ns=2, seed=4)
    full = ds.render_aov(cam, ok)
    ptrs = [full[k].ctypes.data for k in KEYS]
    for q in range(len(KEYS) + 1):
        p = list(ptrs)
        if q < len(KEYS):
            p[q] = None
        bufs = None if q == len(KEYS) else C.byref(rtnw.Aov(*p))
        rc = rtnw.device_lib().rtnw_render_aov(ds.ctx._h, ds._h, C.byref(cam), C.byref(ok), bufs, None)
        assert rc == rtnw.RTNW_ERR_INVALID
    after, _ = ds.render(cam, hs.params(nx=32, ny=32, ns=2, seed=4))
    assert np.array_equal(bits(before), bits(after))


def test_driver_writes_the_aov_files(rtnw, scenes, tmp_path):
    nx, ny, ns = 32, 32, 4
    plain = subprocess.run([str(BIN), "cornell_box", str(nx), str(ny), str(ns), str(tmp_path / "plain.ppm")], capture_output=True, text=True)
    assert plain.returncode == 0, plain.stderr
    r = subprocess.run([str(BIN), "cornell_box", str(nx), str(ny), str(ns), str(tmp_path / "out.ppm"), "--aov", str(tmp_path / "P")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "out.ppm").read_bytes() == (tmp_path / "plain.ppm").read_bytes()
    hs, ds = scenes("cornell_box")
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=1)
    sums, _ = ds.render(cam, params)
    aov = ds.render_aov(cam, params)
    h = aov["hits"].astype(np.float32)
    safe = np.maximum(h, np.float32(1))
    want = dict(color=sums / np.float32(ns), albedo=aov["albedo"] / np.float32(ns),
                normal=np.where(h[..., None] > 0, aov["normal"] / safe[..., None], np.float32(0)),
                depth=np.where(h > 0, aov["depth"] / safe, np.float32(0)))
    for k, v in want.items():
        lines, got = read_pfm(tmp_path / f"P_{k}.pfm")
        assert lines == ["Pf" if k == "depth" else "PF", f"{nx} {ny}", "-1.0"]
        assert np.array_equal(bits(got), bits(v.astype(np.float32))), k
    bad = subprocess.run([str(BIN), "cornell_box", "8", "8", "1", str(tmp_path / "x.ppm"), "--aov", str(tmp_path / "Q"), "--gpus", "2"],
                         capture_output=True, text=True)
    assert bad.returncode != 0 and not (tmp_path / "Q_color.pfm").exists()
