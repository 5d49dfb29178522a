"""Host scene library vs the reference's own builders (CPU only).

The chapter builders of host/scenes/chapter_scenes.cpp are written against the drop-in scene API; flattened, they
must describe object-for-object the scene that the reference's builders (PSC/main.cpp:49-230, compiled unmodified
into oracle/_ref/libref_oracle.so) construct: same leaf order, geometry bits, wrappers, materials, perlin tables.
Without the compiled reference (it needs the original project's sources) the host library is compared with
tests/golden/pinned_scenes.npz (tests/golden/make_pinned_golden.py): leaf counts and SHA-256 digests of the flattened
tables, the perlin tables and the camera origins, recorded where this module held them equal to the reference's objects.
"""
from pathlib import Path

import numpy as np
import pytest

import ref_oracle as ro
from raysets import digest

PINNED = Path(__file__).resolve().parent / "golden" / "pinned_scenes.npz"

SCENES = ["ch01_random", "two_perlin", "cornell_box", "cornell_smoke", "final", "final+bvh", "final_northstar", "earth",
          "simple_light", "two_spheres", "random_scene", "test"]


def _tables(rtnw, hs):
    d = hs.desc
    prims = np.ctypeslib.as_array(d.prims, shape=(d.n_prim_slots,)).view(
        np.dtype([("f", np.float32, 6), ("kx", np.uint32), ("mat", np.int32)]))
    ids = np.ctypeslib.as_array(d.prim_ids, shape=(d.n_prim_slots,))
    xf = np.ctypeslib.as_array(d.xforms, shape=(d.n_xform_ops,)).view(
        np.dtype([("a", np.float32), ("b", np.float32), ("c", np.float32), ("kind", np.uint32)]))
    mats = np.ctypeslib.as_array(d.materials, shape=(d.n_materials,)).view(
        np.dtype([("kind", np.uint32), ("tex", np.int32), ("f", np.float32), ("pad0", np.uint32), ("albedo", np.float32, 3),
                  ("pad1", np.uint32)]))
    texs = np.ctypeslib.as_array(d.textures, shape=(d.n_textures,)).view(
        np.dtype([("kind", np.uint32), ("i0", np.int32), ("i1", np.int32), ("i2", np.int32), ("c", np.float32, 3),
                  ("pad", np.uint32)]))
    return prims, ids, xf, mats, texs


@pytest.mark.parametrize("name", SCENES)
def test_flattened_scene_matches_reference_objects(rtnw, name):
    hs = rtnw.HostScene(name)
    if ro.available():
        rs = ro.RefScene(name, tagged=False)
        assert hs.leaf_count == rs.leaf_count
        dump = rs.dump()
    else:
        p = np.load(PINNED)
        assert hs.leaf_count == int(p[f"leaves:{name}"]) and scene_digest(rtnw, hs) == str(p[f"tables:{name}"])
        dump = None
    prims, ids, xf, mats, texs = _tables(rtnw, hs)
    d = hs.desc
    # item chains apply to BVH leaves of that item
    item_chain = {}
    items = np.ctypeslib.as_array(d.items, shape=(d.n_items,)).view(
        np.dtype([("kind", np.uint32), ("xform", np.uint32), ("first", np.int32), ("count", np.int32), ("bmin", np.float32, 3),
                  ("flip", np.uint32), ("bmax", np.float32, 3), ("pad", np.uint32)]))
    first_slot = {}
    for s in range(d.n_prim_slots):
        if ids[s] >= 0 and ids[s] not in first_slot and (prims[s]["kx"] & 7) != 7:
            first_slot[int(ids[s])] = s
    assert sorted(first_slot) == list(range(hs.leaf_count))
    nodes = np.ctypeslib.as_array(d.nodes, shape=(max(d.n_nodes, 1),)).view(np.dtype([
        ("lmin", np.float32, 3), ("left", np.int32), ("lmax", np.float32, 3), ("right", np.int32), ("rmin", np.float32, 3),
        ("lcount", np.int32), ("rmax", np.float32, 3), ("rcount", np.int32)])) if d.n_nodes else None
    slot_item_chain = np.zeros(d.n_prim_slots, dtype=np.int64)
    for it in items:
        if it["kind"] == 1:  # BVH: collect leaf slots below the root
            stack = [int(it["first"])]
            while stack:
                n = nodes[stack.pop()]
                for ref, cnt in ((n["left"], n["lcount"]), (n["right"], n["rcount"])):
                    if ref == -2**31:
                        continue
                    if ref >= 0:
                        stack.append(int(ref))
                    else:
                        slot_item_chain[~ref:~ref + cnt] = it["xform"]

    def chain_ops(c):
        if c == 0:
            return []
        n = int(xf[c]["kind"]) >> 8
        return [(int(xf[c + k]["kind"]) & 255, float(xf[c + k]["a"]), float(xf[c + k]["b"]), float(xf[c + k]["c"])) for k in range(n)]

    if dump is not None:  # per-leaf comparison with the reference's objects
        for leaf in range(hs.leaf_count):
            s = first_slot[leaf]
            p = prims[s]
            o = dump[leaf]
            kind = int(p["kx"]) & 7
            assert kind == int(o[0]), (leaf, kind, o[0])
            geo = [float(x) for x in p["f"]]
            if kind == 0:
                assert geo[:4] == [float(x) for x in o[1:5]]
            elif kind == 1:
                ext = prims[s + 1]
                assert geo == [float(x) for x in o[1:7]] and [float(x) for x in ext["f"][:3]] == [float(x) for x in o[7:10]]
            elif kind in (2, 3, 4):
                assert geo[:5] == [float(x) for x in o[1:6]]
            elif kind == 5:
                assert geo == [float(x) for x in o[1:7]]
            elif kind == 6:
                assert geo[0] == float(o[1])
            # wrappers of the leaf itself, outermost first (wrappers around a whole bvh_node live on the item, below)
            ops = chain_ops(int(p["kx"]) >> 4)
            nw = int(o[10]) % 100
            flips = int(o[10]) // 100
            assert len(ops) == nw, (leaf, ops, o[10:19])
            assert ((int(p["kx"]) >> 3) & 1) == flips
            for k, op in enumerate(ops[:2]):
                assert op[0] == int(o[11 + 4 * k])
                if op[0] == 1:
                    assert list(op[1:]) == [float(x) for x in o[12 + 4 * k:15 + 4 * k]]
                else:
                    assert list(op[1:3]) == [float(x) for x in o[12 + 4 * k:14 + 4 * k]]
            # material
            m = mats[p["mat"]]
            assert int(m["kind"]) == int(o[19])
            if m["kind"] == 1:
                assert [float(x) for x in m["albedo"]] == [float(x) for x in o[20:23]] and float(m["f"]) == float(o[23])
            elif m["kind"] == 2:
                assert float(m["f"]) == float(o[23])
            else:
                t = texs[m["tex"]]
                if t["kind"] == 0:
                    assert [float(x) for x in t["c"]] == [float(x) for x in o[20:23]]
                elif t["kind"] == 1:
                    assert o[20] == -1
                elif t["kind"] == 2:
                    assert o[20] == -2 and float(t["c"][0]) == float(o[21])
                else:
                    assert o[20] == -3

    if name == "final_northstar":  # translate(rotate_y(bvh_node(spheres), 15), (-100,270,395)), SURVEY.md §8d item 5
        assert [int(k) for k in items["kind"]] == [1, 0, 1]
        assert chain_ops(int(items[0]["xform"])) == []
        ops = chain_ops(int(items[2]["xform"]))
        assert [o[0] for o in ops] == [1, 2] and ops[0][1:] == (-100.0, 270.0, 395.0)
        rad = np.float32((np.pi / 180.0) * 15.0)
        assert abs(ops[1][1] - np.sin(np.float64(rad))) < 1e-7 and abs(ops[1][2] - np.cos(np.float64(rad))) < 1e-7
        assert set(slot_item_chain[slot_item_chain > 0]) == {int(items[2]["xform"])}


def test_perlin_tables_match_reference(rtnw):
    hs = rtnw.HostScene("two_perlin")
    if ro.available():
        ro.RefScene("two_perlin", tagged=False)  # regenerates the reference's static tables from the same drand48 state
        rv, px, py, pz = ro.perlin_tables()
    else:
        p = np.load(PINNED)
        rv, px, py, pz = (p[f"perlin_{k}"] for k in ("ranvec", "perm_x", "perm_y", "perm_z"))
    d = hs.desc
    assert np.array_equal(np.ctypeslib.as_array(d.perlin_ranvec, shape=(768,)), rv)
    assert np.array_equal(np.ctypeslib.as_array(d.perlin_perm_x, shape=(256,)), px)
    assert np.array_equal(np.ctypeslib.as_array(d.perlin_perm_y, shape=(256,)), py)
    assert np.array_equal(np.ctypeslib.as_array(d.perlin_perm_z, shape=(256,)), pz)


def test_camera_matches_reference_constructor(rtnw):
    # the reference camera is private; its get_ray with aperture 0 exposes origin and the affine map (s,t) -> direction
    for name in ["ch01_random", "final"]:
        hs = rtnw.HostScene(name)
        v = ro.view_of(name)
        v0 = dict(v, aperture=0.0)
        nx, ny = 200, 100
        origin = ro.camera_rays(v0, nx, ny, [[0, 0], [nx - 1, ny - 1]], [0, 0], seed=3)["origin"][0] if ro.available() \
            else np.load(PINNED)[f"camera_origin:{name}"]
        cam = rtnw.make_camera(v["lookfrom"], v["lookat"], v["vfov"], nx / ny, 0.0, 10.0, 0.0, 1.0)
        assert np.array_equal(origin, np.array(cam.origin, dtype=np.float32))
        cam2 = hs.camera(nx, ny)
        assert list(cam2.lower_left_corner) == list(cam.lower_left_corner)
        assert list(cam2.horizontal) == list(cam.horizontal) and list(cam2.vertical) == list(cam.vertical)


def scene_digest(rtnw, hs) -> str:
    """the flattened tables of a host scene, byte for byte (items, BVH nodes, prim slots and ids, transforms, materials,
    textures, texture images)"""
    import ctypes as C
    d = hs.desc

    def arr(ptr, n, ctype):
        return np.frombuffer(C.string_at(ptr, n * C.sizeof(ctype)), dtype=np.uint8) if n else np.zeros(0, np.uint8)
    return digest(arr(d.items, d.n_items, rtnw.Item), arr(d.nodes, d.n_nodes, rtnw.BvhNode), arr(d.prims, d.n_prim_slots, rtnw.Prim),
                  arr(d.prim_ids, d.n_prim_slots, C.c_int32), arr(d.xforms, d.n_xform_ops, rtnw.XformOp),
                  arr(d.materials, d.n_materials, rtnw.Material), arr(d.textures, d.n_textures, rtnw.Texture),
                  arr(d.images, int(d.image_bytes), C.c_uint8))
