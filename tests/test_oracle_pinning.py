"""Pins the C restatement (oracle/rtnw_oracle.c, run on the flattened tables of the host library) against the reference
renderer itself (oracle/_ref/libref_oracle.so = the reference's sources compiled unmodified + F2 fix).  CPU only.

Same compiler, same libm, same sample stream => everything is required to be BIT-EXACT, whole images included.
Without the compiled reference (it needs the original project's sources) the same outputs are compared with
tests/golden/pinned_port.npz (tests/golden/make_pinned_golden.py): the restatement's outputs for exactly these cases,
recorded where this module held them bit-exact to the reference — arrays for renders and camera rays, SHA-256 digests of
the bytes for hits, texture values and scatter results."""
from pathlib import Path

import numpy as np
import pytest

import oracle_port as op
import ref_oracle as ro
from raysets import FLT_MAX, assert_hits_equal, digest, make_rays

PINNED = Path(__file__).resolve().parent / "golden" / "pinned_port.npz"
T_RANGES = [(0.001, FLT_MAX), (0.0, 500.0)]


def pinned():
    return np.load(PINNED)

SCENES = ["ch01_random", "two_perlin", "cornell_box", "cornell_smoke", "final", "final+bvh", "final_northstar", "earth",
          "simple_light", "random_scene", "test", "random_scene+bvh", "ch01_random+bvh", "cornell_box+bvh", "cornell_smoke+bvh"]


@pytest.mark.parametrize("name", SCENES)
def test_port_closest_hit_bit_exact(rtnw, name):
    rs, rays, got = trace_outputs(rtnw, name)
    if not ro.available():
        assert digest(rays, *got) == str(pinned()[f"trace:{name}"])
        return
    for (t_min, t_max), g in zip(T_RANGES, got):
        assert_hits_equal(g, rs.trace(rays, t_min, t_max, seed=11), uv_tol=0)


def trace_outputs(rtnw, name):
    rs, rays = make_rays(name, n_primary=1200, rtnw=rtnw)
    hs = rtnw.HostScene(name)
    return rs, rays, [op.trace(rtnw, hs.desc_ptr, rays, t_min, t_max, seed=11) for t_min, t_max in T_RANGES]


RENDER_CASES = [("ch01_random", 48, 24, 4), ("two_perlin", 48, 24, 4), ("cornell_box", 32, 32, 6),
                ("cornell_smoke", 32, 32, 6), ("final", 24, 24, 2), ("final+bvh", 32, 32, 3),
                ("final_northstar", 32, 32, 3), ("simple_light", 32, 16, 4), ("earth", 24, 24, 3), ("random_scene", 40, 20, 4), ("test", 32, 16, 4), ("two_spheres", 24, 24, 4),
                ("perlin_v1", 40, 20, 4), ("perlin_v2", 40, 20, 4), ("perlin_v3", 40, 20, 4),
                ("cornell_smoke:ch08", 24, 24, 4), ("random_scene:ch03", 40, 20, 4)]


def render_outputs(rtnw, name, nx, ny, ns):
    hs = rtnw.HostScene(name)
    return op.render(rtnw, hs.desc_ptr, hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=99))


@pytest.mark.parametrize("name,nx,ny,ns", RENDER_CASES)
def test_port_render_bit_exact(rtnw, name, nx, ny, ns):
    got, st = render_outputs(rtnw, name, nx, ny, ns)
    if ro.available():
        want, rst = ro.RefScene(name, tagged=True).render(nx, ny, ns, seed=99, rng_mode=1)
    else:
        p = pinned()
        want, rst = p[f"render:{name}"], dict(zip(("rays", "aabb"), p[f"render_stats:{name}"].tolist()))
    same = (got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))
    assert same.all(), f"{(~same).sum()} of {same.size} sums differ, max {np.nanmax(np.abs(got - want))}"
    assert st["rays"] == rst["rays"] and st["paths"] == nx * ny * ns
    if "bvh" in name or name == "final_northstar":
        assert st["box_tests"] == rst["aabb"]


def test_port_sample_split_and_camera(rtnw):
    hs = rtnw.HostScene("ch01_random")
    nx, ny = 40, 20
    cam = hs.camera(nx, ny)
    rng = np.random.default_rng(0)
    ij = np.stack([rng.integers(0, nx, 500), rng.integers(0, ny, 500)], axis=1)
    s = rng.integers(0, 100, 500)
    got = op.camera_rays(rtnw, cam, nx, ny, ij, s, seed=5)
    want = ro.camera_rays(ro.view_of("ch01_random"), nx, ny, ij, s, seed=5) if ro.available() else pinned()["camera_rays"]
    for f in ("origin", "direction", "time", "key"):
        assert np.array_equal(got[f], want[f]), f
    full, _ = op.render(rtnw, hs.desc_ptr, cam, hs.params(nx=nx, ny=ny, ns=4, seed=3))
    parts = sum(op.render(rtnw, hs.desc_ptr, cam, hs.params(nx=nx, ny=ny, ns=2, seed=3, sample_begin=g, sample_stride=2))[0]
                .astype(np.float64) for g in range(2))
    assert np.allclose(parts, full, rtol=1e-6, atol=1e-6)


def unit_outputs(rtnw):
    """[(key, the restatement's outputs, a callable giving the reference's)] for perlin, the textures and scatter"""
    rng = np.random.default_rng(2)
    hs = rtnw.HostScene("two_perlin")
    xyz = np.concatenate([rng.normal(scale=3, size=(2000, 3)), rng.normal(scale=400, size=(2000, 3))]).astype(np.float32)
    out = [(f"perlin{which}", (op.eval_perlin(rtnw, hs.desc_ptr, which, xyz),), lambda which=which: (ro.eval_perlin(which, xyz),))
           for which in (0, 1)]
    uvp = np.concatenate([rng.random((len(xyz), 2)).astype(np.float32), xyz], axis=1)
    d = hs.desc
    kinds = [d.textures[i].kind for i in range(d.n_textures)]
    out.append(("checker", (op.eval_texture(rtnw, hs.desc_ptr, kinds.index(1), uvp),),
                lambda: (ro.eval_texture(1, [0.2, 0.3, 0.1, 0.9, 0.9, 0.9], uvp),)))
    out.append(("noise", (op.eval_texture(rtnw, hs.desc_ptr, kinds.index(2), uvp),), lambda: (ro.eval_texture(2, [4.0], uvp),)))
    he = rtnw.HostScene("earth")
    ke = [he.desc.textures[i].kind for i in range(he.desc.n_textures)]
    out.append(("image", (op.eval_texture(rtnw, he.desc_ptr, ke.index(3), uvp),), lambda: (ro.eval_texture(3, [], uvp),)))
    # scatter through the materials of the final scene: lambertian(const), dielectric, metal, light, isotropic, lambertian(noise)
    hf = rtnw.HostScene("final")
    df = hf.desc
    n = 600
    rays = np.zeros(n, dtype=rtnw.RAY_DTYPE)
    rays["origin"] = rng.normal(size=(n, 3)); rays["direction"] = rng.normal(size=(n, 3)); rays["time"] = rng.random(n)
    hits = np.zeros(n, dtype=rtnw.HIT_DTYPE)
    nrm = rng.normal(size=(n, 3)); hits["normal"] = nrm / np.linalg.norm(nrm, axis=1, keepdims=True)
    hits["p"] = rng.normal(scale=100, size=(n, 3)); hits["t"] = 1; hits["u"] = rng.random(n); hits["v"] = rng.random(n)
    for m in range(df.n_materials):
        mt = df.materials[m]
        tex = df.textures[mt.tex] if mt.tex >= 0 else None
        if tex is not None and tex.kind not in (0, 2):
            continue
        h = hits.copy()
        h["mat_id"] = m
        row = [mt.kind, 2 if (tex is not None and tex.kind == 2) else 0] + \
              (list(tex.c) if (tex is not None and tex.kind == 0) else list(mt.albedo)) + [mt.f, tex.c[0] if (tex is not None and tex.kind == 2) else 0, 0]
        out.append((f"scatter{m}", op.scatter(rtnw, hf.desc_ptr, rays, h, seed=8),
                    lambda row=row, h=h: ro.scatter(np.tile(np.array(row, dtype=np.float32), (n, 1)), rays, h, seed=8)))
    return out


def test_port_textures_perlin_scatter(rtnw):
    outs = unit_outputs(rtnw)
    if not ro.available():
        p = pinned()
        for key, got, _ in outs:
            assert digest(*got) == str(p[f"unit:{key}"]), key
        return
    ro.RefScene("two_perlin", tagged=False)
    for key, got, want in outs:
        for a, b in zip(got, want()):
            if a.dtype.names:
                for f in ("origin", "direction", "time"):
                    assert np.array_equal(a[f], b[f], equal_nan=True), (key, f)
            else:
                assert np.array_equal(a, b, equal_nan=key.startswith("scatter")), key
