"""Deterministic ray sets shared by the parity tests and the golden-fixture generator, and the reference side those tests
compare with: the compiled reference (oracle/_ref/libref_oracle.so) when it is built, otherwise the C restatement
(oracle/rtnw_oracle.c).  Without the compiled reference, the restatement is held on every run to stored data only:
  * tests/test_golden.py: bit for bit against the fixtures generated from the reference itself (hits of 13 scenes, small
    renders of 15, perlin / texture / camera / scatter values);
  * tests/test_oracle_pinning.py: bit for bit against its own outputs recorded where that module held them equal to the
    reference (hits of 15 scenes, random_scene among them, and 17 small renders; tests/golden/pinned_port.npz).
Cases outside those sets, such as the full-size renders of tests/test_gpu_parity.py, rest on the restatement computing
them with the same code paths."""
import hashlib

import numpy as np

import oracle_port as op
import ref_oracle as ro

FLT_MAX = float(np.finfo(np.float32).max)


class PortScene:
    """RefScene's trace / render (tagged leaves, the shared Philox sample stream) computed by the C restatement"""

    def __init__(self, rtnw, name):
        self.rtnw, self.hs = rtnw, rtnw.HostScene(name)

    def trace(self, rays, t_min=0.001, t_max=FLT_MAX, seed=1):
        return op.trace(self.rtnw, self.hs.desc_ptr, rays, t_min, t_max, seed=seed)

    def render(self, nx, ny, ns, seed=1, rng_mode=1):
        assert rng_mode == 1, "the C restatement draws from the shared Philox stream only"
        return op.render(self.rtnw, self.hs.desc_ptr, self.hs.camera(nx, ny), self.hs.params(nx=nx, ny=ny, ns=ns, seed=seed))


def reference_scene(rtnw, name):
    return ro.RefScene(name, tagged=True) if ro.available() else PortScene(rtnw, name)


def reference_camera_rays(rtnw, name, nx, ny, ij, sample, seed=1):
    if ro.available():
        return ro.camera_rays(ro.view_of(name), nx, ny, ij, sample, seed=seed)
    return op.camera_rays(rtnw, rtnw.HostScene(name).camera(nx, ny), nx, ny, ij, sample, seed=seed)


def make_rays(name, n_primary=3000, seed=7, rtnw=None):
    """primary camera rays + secondary rays leaving real hit points + stress rays (axis-parallel, zero components,
    origins inside the scene volume).  Returns (reference scene, rays); pass the package as `rtnw` to fall back to the
    C restatement when the compiled reference is absent."""
    rng = np.random.default_rng(seed)
    nx, ny = 120, 90
    ij = np.stack([rng.integers(0, nx, n_primary), rng.integers(0, ny, n_primary)], axis=1)
    prim = reference_camera_rays(rtnw, name, nx, ny, ij, rng.integers(0, 50, n_primary), seed=seed)
    rs = reference_scene(rtnw, name)
    h = rs.trace(prim, 0.001, FLT_MAX, seed=seed)
    hit = h["prim_id"] >= 0
    sec = np.zeros(int(hit.sum()) * 2, dtype=ro.RAY_DTYPE)
    p = np.repeat(h["p"][hit], 2, axis=0)
    d = rng.normal(size=p.shape).astype(np.float32)
    d[::2] = d[::2] + h["normal"][hit]  # half of them lambertian-like
    sec["origin"] = p
    sec["direction"] = d
    sec["time"] = rng.random(len(sec)).astype(np.float32)
    sec["key"] = rng.integers(0, 2**31, len(sec), dtype=np.uint32)
    lo, hi = h["p"][hit].min(axis=0) - 1, h["p"][hit].max(axis=0) + 1
    m = max(n_primary // 2, 16)
    st = np.zeros(m, dtype=ro.RAY_DTYPE)
    st["origin"] = (lo + rng.random((m, 3)) * (hi - lo)).astype(np.float32)
    dd = rng.normal(size=(m, 3)).astype(np.float32)
    dd[np.arange(m), rng.integers(0, 3, m)] *= (rng.random(m) < 0.5)  # zero one component in half of them
    axis = rng.random(m) < 0.25
    dd[axis] = np.eye(3, dtype=np.float32)[rng.integers(0, 3, int(axis.sum()))] * rng.choice([-1.0, 1.0], int(axis.sum()))[:, None]
    st["direction"] = dd
    st["time"] = rng.random(m).astype(np.float32)
    st["key"] = rng.integers(0, 2**31, m, dtype=np.uint32)
    return rs, np.concatenate([prim, sec, st])


def digest(*arrays) -> str:
    """SHA-256 of the arrays' bytes: a bit-exact stored stand-in for outputs too large to keep under tests/golden/"""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def assert_hits_equal(got, want, uv_tol=1e-5):
    """leaf ids / faces exact; t, p, normal bit-exact (NaN-aware); u, v within uv_tol (0 = bit-exact)"""
    assert np.array_equal(got["prim_id"], want["prim_id"]), f"{(got['prim_id'] != want['prim_id']).sum()} leaf ids differ"
    hit = want["prim_id"] >= 0
    assert np.array_equal(got["sub_id"][hit], want["sub_id"][hit])
    for f in ("t", "p", "normal"):
        a, b = got[f][hit], want[f][hit]
        same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b)) | ((a == 0) & (b == 0))
        assert same.all(), f"{f}: {(~same).sum()} of {same.size} values differ, max abs {np.nanmax(np.abs(a - b))}"
    for f in ("u", "v"):
        a, b = got[f][hit], want[f][hit]
        ok = (a == b) | (np.isnan(a) & np.isnan(b)) if uv_tol == 0 else np.isclose(a, b, rtol=uv_tol, atol=uv_tol) | (np.isnan(a) & np.isnan(b))
        assert ok.all(), f"{f}: max abs diff {np.nanmax(np.abs(a - b))}"


def scene_with_material(rtnw, kind, rgb, f, scale=0.0):
    """a one-sphere scene_desc whose material 0 is the requested one (tables built by hand through the C structs)"""
    import ctypes as C
    hs = rtnw.HostScene("two_perlin")  # borrow perlin tables / xform identity
    d = rtnw.SceneDesc()
    C.memmove(C.byref(d), C.byref(hs.desc), C.sizeof(d))
    tex = (rtnw.Texture * 1)()
    tex[0].kind = 2 if scale else 0
    tex[0].c[0], tex[0].c[1], tex[0].c[2] = (scale, 0, 0) if scale else rgb
    mat = (rtnw.Material * 1)()
    mat[0].kind = kind
    mat[0].tex = 0
    mat[0].f = f
    mat[0].albedo[0], mat[0].albedo[1], mat[0].albedo[2] = rgb
    prim = (rtnw.Prim * 1)()
    prim[0].f[3] = 1.0
    prim[0].kx = 0
    prim[0].mat = 0
    ids = (C.c_int32 * 1)(0)
    item = (rtnw.Item * 1)()
    item[0].kind, item[0].first, item[0].count = 0, 0, 1
    d.n_items, d.items = 1, item
    d.n_nodes = 0
    d.n_prim_slots, d.prims, d.prim_ids = 1, prim, ids
    d.n_materials, d.materials = 1, mat
    d.n_textures, d.textures = 1, tex
    keep = (hs, tex, mat, prim, ids, item)
    return d, keep
