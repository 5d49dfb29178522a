"""The device tables rtnw_scene_upload builds (record stream, gates, 4-wide gate tree), checked on the CPU through
rtnw_scene_inspect — no GPU.  DESIGN.md §3 rests the traversal's exactness on three properties of these tables:
  1. every leaf of a reference bvh_node hangs under exactly one gate, every gate under exactly one wide-node slot;
  2. interior boxes of the gate tree are EXACT float unions of what is beneath them;
  3. therefore (IEEE monotonicity of the slab test) walking the gate tree reaches exactly the gates whose own box passes
     aabb::hit — the set the reference's bvh_node::hit reaches.  Property 3 is tested directly, in float32, on random,
     axis-parallel, zero-component and on-plane rays."""
import importlib
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")

NONE = -2**31
K_MSPHERE, K_MEDIUM, K_EXT, K_ITEM, K_END = 1, 6, 7, 9, 10
TAG_LAST = 64
SCENES = ["final_northstar", "final+bvh", "ch01_random+bvh", "cornell_smoke+bvh", "stress_shells+bvh"]


def _tables(name):
    hs = rtnw.HostScene(name)
    t = rtnw.device_tables(hs.desc_ptr)
    t["tag"] = t["recs"][:, 6].copy().view(np.uint32)
    t["ival"] = t["recs"][:, 7].copy().view(np.int32)
    t["ref"] = t["wnodes"][:, 24:28].copy().view(np.int32)
    return hs, t


def _items(t, fast=False):
    """(record index, next, root, depth, is_bvh) of the top-level list's items; fast=True: root / depth of the tree over the
    leaves' own boxes (RTNW_F_FAST_BVH) instead of the gate tree"""
    out, i = [], 0
    while (t["tag"][i] & 15) == K_ITEM:
        a = t["recs"][i, :5].copy().view(np.int32)
        out.append((i, int(a[0]), int(a[3] if fast else a[1]), int(a[4] if fast else a[2]), int(t["ival"][i]) == 1))
        i = int(a[0])
    assert (t["tag"][i] & 15) == K_END and i == len(t["recs"]) - 1
    return out


def _child_box(t, n, j):
    w = t["wnodes"][n]
    return w[[j, 4 + j, 8 + j]], w[[12 + j, 16 + j, 20 + j]]


def _subtree(t, n, depth, gates_seen, nodes_seen):
    """exact union box of wide node n; records which gates / nodes hang under it; returns (min, max, depth)"""
    assert n not in nodes_seen, "wide node referenced twice"
    nodes_seen.add(n)
    lo, hi, deepest = None, None, depth
    for j in range(4):
        r = int(t["ref"][n, j])
        if r == NONE:
            continue
        bmin, bmax = _child_box(t, n, j)
        if r >= 0:
            cmin, cmax, d = _subtree(t, r, depth + 1, gates_seen, nodes_seen)
            # property 2: the stored box of an interior child is the exact union of its children's boxes
            assert np.array_equal(bmin, cmin) and np.array_equal(bmax, cmax), (n, j)
            deepest = max(deepest, d)
        else:
            g = ~r
            assert 0 <= g < len(t["gates"]) and g not in gates_seen, "gate referenced twice"
            gates_seen.add(g)
        lo = bmin if lo is None else np.fmin(lo, bmin)
        hi = bmax if hi is None else np.fmax(hi, bmax)
    assert lo is not None, "empty wide node"
    return lo, hi, deepest


def _leaf_records(t, first):
    """records a leaf scan starting at `first` tests (test_leaf in rtnw_device.cuh): up to and including the LAST tag"""
    out, i = [], first
    while True:
        kind = int(t["tag"][i] & 15)
        assert kind < K_EXT or kind == K_MEDIUM, (i, kind)
        out.append(i)
        step = 2 if kind == K_MSPHERE else (1 + int(t["recs"][i, 2:3].copy().view(np.int32)[0]) if kind == K_MEDIUM else 1)
        if t["tag"][i] & TAG_LAST:
            return out, i + step
        i += step


@pytest.mark.parametrize("name", SCENES)
def test_gates_and_gate_tree_structure(name):
    hs, t = _tables(name)
    gates_seen, nodes_seen, covered = set(), set(), set()
    for i, nxt, root, depth, is_bvh in _items(t):
        if not is_bvh:
            continue
        before = set(gates_seen)
        _, _, deepest = _subtree(t, root, 1, gates_seen, nodes_seen)
        assert deepest <= depth, "the recorded tree depth (stack reserve) is too small"
        for g in sorted(gates_seen - before):
            l0, l1 = (int(x) for x in t["gates"][g])
            assert l0 > i and l0 < nxt and (l1 == -1 or i < l1 < nxt)
            recs0, end0 = _leaf_records(t, l0)
            if l1 >= 0:  # the two leaf children of one bvh_node are neighbours in left-to-right order
                assert l1 == end0
                recs1, _ = _leaf_records(t, l1)
            else:
                recs1 = []
            for r in recs0 + recs1:
                assert r not in covered, "a record is tested through two gates"
                covered.add(r)
        # every primitive head record of the item belongs to exactly one gate's leaves
        j = i + 1
        while j < nxt:
            kind = int(t["tag"][j] & 15)
            assert j in covered, (name, j)
            j += 2 if kind == K_MSPHERE else (1 + int(t["recs"][j, 2:3].copy().view(np.int32)[0]) if kind == K_MEDIUM else 1)
    # the second tree of every BVH item (RTNW_F_FAST_BVH): one gate per leaf behind the leaf's own (padded) box, every leaf
    # exactly once, interior boxes again exact unions; both trees together use every gate and every wide node of the tables
    fast_gates, fast_leaves = set(), set()
    for i, nxt, root, depth, is_bvh in _items(t, fast=True):
        if not is_bvh:
            continue
        mine = set()
        _, _, deepest = _subtree(t, root, 1, mine, nodes_seen)
        assert deepest <= depth and not (mine & gates_seen) and not (mine & fast_gates)
        for g in mine:
            l0, l1 = (int(x) for x in t["gates"][g])
            assert l1 == -1 and i < l0 < nxt and l0 not in fast_leaves
            fast_leaves.add(l0)
        fast_gates |= mine
    exact_leaves = set()
    for g in gates_seen:
        l0, l1 = (int(x) for x in t["gates"][g])
        exact_leaves |= {l0} | ({l1} if l1 >= 0 else set())
    assert hs.desc.n_nodes == 0 or fast_leaves == exact_leaves
    assert (gates_seen | fast_gates) == set(range(len(t["gates"]))) or (len(t["gates"]) == 1 and int(t["gates"][0, 0]) == -1)
    assert nodes_seen == set(range(len(t["wnodes"])))
    assert hs.desc.n_nodes == 0 or len(gates_seen) > 0


def _hit_aabb(bmin, bmax, o, inv, t_lo, t_hi):
    """aabb::hit with r.origin() (PSC/aabb.h:33-49 + F2) in float32, as the node tasks of coop_bvh_item (rtnw_device.cuh)
    evaluate it; boxes: (n,3)"""
    lo = np.full(len(bmin), t_lo, dtype=np.float32)
    hi = np.full(len(bmin), t_hi, dtype=np.float32)
    with np.errstate(all="ignore"):
        for a in range(3):
            near = bmax[:, a] if inv[a] < 0 else bmin[:, a]
            far = bmin[:, a] if inv[a] < 0 else bmax[:, a]
            t0 = (near - o[a]) * inv[a]
            t1 = (far - o[a]) * inv[a]
            lo = np.fmax(t0, lo)  # NaN-ignoring, like fmaxf
            hi = np.fmin(t1, hi)
    return ~(hi <= lo) | np.isnan(np.float32(t_hi))


def _rays(rng, lo, hi, n):
    """rays aimed at points inside [lo, hi] from origins around it, then made degenerate in the ways that stress the slab test"""
    span = (hi - lo).astype(np.float32)
    o = (lo - span + rng.random((n, 3), dtype=np.float32) * 3 * span).astype(np.float32)
    target = (lo + rng.random((n, 3), dtype=np.float32) * span).astype(np.float32)
    d = (target - o).astype(np.float32)
    k = n // 8
    d[:k, rng.integers(0, 3)] = 0.0                      # a zero direction component
    axis = rng.integers(0, 3, size=k)                    # axis-parallel, through the target
    d[k:2 * k] = 0.0
    d[np.arange(k, 2 * k), axis] = np.where(rng.random(k) < 0.5, -1.5, 1.5).astype(np.float32)
    o[k:2 * k] = target[k:2 * k] - d[k:2 * k] * np.float32(2.0) * span.max()
    d[2 * k:3 * k] *= np.float32(1e-6)                   # tiny directions: large 1/d
    o[3 * k:4 * k, 0] = lo[0]                            # origins on a bounding plane
    o[4 * k:5 * k] = (lo + rng.random((k, 3), dtype=np.float32) * span).astype(np.float32)  # origins inside
    d[5 * k:6 * k, 1] = -0.0                             # negative zero
    o[5 * k:6 * k, 1] = target[5 * k:6 * k, 1]
    return o, d


@pytest.mark.parametrize("name", SCENES)
def test_gate_tree_walk_reaches_exactly_the_gates_whose_box_passes(name):
    """property 3 (the reference's leaf set): in float32, for every ray and both a wide and a narrow t range"""
    hs, t = _tables(name)
    rng = np.random.default_rng(len(name))
    for i, nxt, root, depth, is_bvh in _items(t):
        if not is_bvh:
            continue
        # all (gate, box) pairs and all interior (node, box) pairs under this root
        gate_box, stack, nodes = {}, [root], []
        while stack:
            n = stack.pop()
            nodes.append(n)
            for j in range(4):
                r = int(t["ref"][n, j])
                if r == NONE:
                    continue
                if r >= 0:
                    stack.append(r)
                else:
                    gate_box[~r] = _child_box(t, n, j)
        ids = np.array(sorted(gate_box))
        gmin = np.stack([gate_box[g][0] for g in ids]).astype(np.float32)
        gmax = np.stack([gate_box[g][1] for g in ids]).astype(np.float32)
        o_all, d_all = _rays(rng, gmin.min(0), gmax.max(0), 240)
        n_hit = 0
        for o, d in zip(o_all, d_all):
            with np.errstate(all="ignore"):
                inv = (np.float32(1.0) / d).astype(np.float32)
            for t_lo, t_hi in ((0.001, 3.0e38), (0.001, float(np.float32(0.6) * np.linalg.norm(gmax.max(0) - gmin.min(0)) / max(np.linalg.norm(d), 1e-20)))):
                brute = set(ids[_hit_aabb(gmin, gmax, o, inv, np.float32(t_lo), np.float32(t_hi))].tolist())
                walked, stack = set(), [root]
                while stack:
                    n = stack.pop()
                    w = t["wnodes"][n]
                    ok = _hit_aabb(w[0:12].reshape(3, 4).T, w[12:24].reshape(3, 4).T, o, inv, np.float32(t_lo), np.float32(t_hi))
                    for j in range(4):
                        r = int(t["ref"][n, j])
                        if r == NONE or not ok[j]:
                            continue
                        if r >= 0:
                            stack.append(r)
                        else:
                            walked.add(~r)
                assert walked == brute, (name, o, d, t_hi, sorted(brute - walked)[:5], sorted(walked - brute)[:5])
                n_hit += len(brute) > 0
        assert n_hit >= 200, "the ray set hardly touches this tree"


def test_inspect_rejects_bad_input():
    hs = rtnw.HostScene("cornell_box")
    assert rtnw.device_lib().rtnw_scene_inspect(hs.desc_ptr, 9, None, 0) < 0
    assert rtnw.device_lib().rtnw_scene_inspect(None, 0, None, 0) < 0
    t = rtnw.device_tables(hs.desc_ptr)  # a scene without a BVH: placeholder gate / node, records only
    assert len(t["recs"]) > 8 and (t["tag"] if "tag" in t else t["recs"][:, 6].view(np.uint32))[-1] & 15 == K_END


@pytest.mark.parametrize("name", ["final_northstar", "cornell_smoke", "final"])
def test_medium_records_carry_the_negated_reciprocal_density(name):
    """PSC/constant_medium.h:42 computes -(1/density) in float for every sample; the upload rounds it once on the host
    (IEEE float division, the same bits) and the kernels multiply by it: A.w of a medium record == -(1.0f / A.x)."""
    _, t = _tables(name)
    med = np.flatnonzero((t["tag"] & 15) == K_MEDIUM)
    assert len(med) >= 2
    rho = t["recs"][med, 0].astype(np.float32)
    want = -(np.float32(1.0) / rho)
    assert np.array_equal(t["recs"][med, 3].view(np.uint32), want.view(np.uint32)), (rho, t["recs"][med, 3])
