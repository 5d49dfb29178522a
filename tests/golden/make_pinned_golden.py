#!/usr/bin/env python
"""Record tests/golden/pinned_port.npz and tests/golden/pinned_scenes.npz: what tests/test_oracle_pinning.py and
tests/test_scene_parity.py compare with, for runs where the compiled reference cannot be built (it needs the original
project's sources, which are not part of this repository).

The values are the outputs of the C restatement (oracle/rtnw_oracle.c) and the host library's flattened scenes as of
commit 5a19849.  At that commit those two modules held exactly these outputs bit-exact to the reference: its hits,
renders, camera rays, texture / perlin / scatter values, and its scene objects and perlin tables.  Large outputs are kept
as SHA-256 digests of their bytes (raysets.digest).  Regenerate only together with a passing run of both modules against
the compiled reference.

    python tests/golden/make_pinned_golden.py        # after __graft_entry__.build()
"""
import importlib
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path[:0] = [str(HERE.parent.parent), str(HERE.parent)]
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")
import oracle_port as op  # noqa: E402
import ref_oracle as ro  # noqa: E402
import test_oracle_pinning as tp  # noqa: E402
import test_scene_parity as ts  # noqa: E402
from raysets import digest  # noqa: E402


def main():
    port = {}
    for name in tp.SCENES:
        _, rays, got = tp.trace_outputs(rtnw, name)
        port[f"trace:{name}"] = digest(rays, *got)
    for name, nx, ny, ns in tp.RENDER_CASES:
        got, st = tp.render_outputs(rtnw, name, nx, ny, ns)
        port[f"render:{name}"] = got
        port[f"render_stats:{name}"] = np.array([st["rays"], st["box_tests"]])
    # the camera rays of test_port_sample_split_and_camera
    nx, ny = 40, 20
    rng = np.random.default_rng(0)
    ij = np.stack([rng.integers(0, nx, 500), rng.integers(0, ny, 500)], axis=1)
    s = rng.integers(0, 100, 500)
    port["camera_rays"] = op.camera_rays(rtnw, rtnw.HostScene("ch01_random").camera(nx, ny), nx, ny, ij, s, seed=5)
    for key, got, _ in tp.unit_outputs(rtnw):
        port[f"unit:{key}"] = digest(*got)
    np.savez_compressed(HERE / "pinned_port.npz", **port)

    scenes = {}
    for name in ts.SCENES:
        hs = rtnw.HostScene(name)
        scenes[f"leaves:{name}"] = hs.leaf_count
        scenes[f"tables:{name}"] = ts.scene_digest(rtnw, hs)
    hp = rtnw.HostScene("two_perlin")  # keeps the tables alive while they are copied
    d = hp.desc
    scenes["perlin_ranvec"] = np.ctypeslib.as_array(d.perlin_ranvec, shape=(768,)).copy()
    for k in ("x", "y", "z"):
        scenes[f"perlin_perm_{k}"] = np.ctypeslib.as_array(getattr(d, f"perlin_perm_{k}"), shape=(256,)).copy()
    for name in ("ch01_random", "final"):  # the cameras of test_camera_matches_reference_constructor
        v = ro.view_of(name)
        cam = rtnw.make_camera(v["lookfrom"], v["lookat"], v["vfov"], 200 / 100, 0.0, 10.0, 0.0, 1.0)
        scenes[f"camera_origin:{name}"] = np.array(cam.origin, dtype=np.float32)
    np.savez_compressed(HERE / "pinned_scenes.npz", **scenes)
    print({p.name: p.stat().st_size for p in (HERE / "pinned_port.npz", HERE / "pinned_scenes.npz")})


if __name__ == "__main__":
    main()
