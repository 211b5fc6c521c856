"""The host side of scene commit that replaces `BVHNode::new` (bvh.rs:54-103), on the CPU: the binned-SAH binary tree
(csrc/bvh.cpp) and its SAH-optimal collapse into the compressed 8-wide tree (csrc/bvh8.cpp), through the host-only entry
point rt1w_build_bvh_host.  Structure (every primitive in exactly one leaf / one leaf slot, children adjacent, depth within
the traversal stacks), conservativeness (every node box contains its subtree; every quantised child box, decoded the way
kernels.cuh: wide_visit decodes it, contains the child's f32 box) and a reference walk in numpy: on both trees the set of
leaves a ray's slab test reaches contains every primitive box the ray really enters (so no closest hit can be culled)."""
import numpy as np
import pytest

from common import check_binary, check_walks, check_wide


def _boxes(api, name, **kw):
    hs = api.HostScene(name, seed=1, **kw)
    prims = api.lower_prims(hs.desc)
    lo = np.array([list(p.bbox_min) for p in prims])
    hi = np.array([list(p.bbox_max) for p in prims])
    ok = np.isfinite(lo).all(1) & np.isfinite(hi).all(1)
    return lo[ok], hi[ok]


def _random_boxes(n, seed):
    rng = np.random.Generator(np.random.Philox(seed))
    c = rng.uniform(-100, 100, (n, 3))
    r = rng.uniform(0.05, 3.0, (n, 3))
    return c - r, c + r


CASES = [("random_scene", {}), ("final_scene", {}), ("stress", dict(stress_spheres=20_000)), ("random boxes", 5000), ("two boxes", 2), ("one box", 1)]


@pytest.mark.parametrize("name,arg", CASES)
def test_host_trees(rt, name, arg):
    api = rt.api
    lo, hi = _random_boxes(arg, 7) if isinstance(arg, int) else _boxes(api, name, **arg)
    t = api.build_bvh_host(lo, hi)
    n_nodes = check_binary(t, lo, hi)
    assert n_nodes == 2 * len(lo) - 1 and len(t["nodes"]) == (2 * len(lo) if len(lo) > 1 else 2)  # + the padding node 1
    fill = check_wide(t, lo, hi)
    print(f"[host bvh] {name}: {len(lo)} boxes -> {len(t['nodes'])} binary nodes (depth {t['depth']}), {len(t['wide_nodes'])} wide nodes "
          f"(depth {t['wide_depth']}, {fill:.2f} slots per node)")
    if len(lo) > 100:
        assert len(t["wide_nodes"]) < 0.45 * len(lo) and fill > 3.0
    # reference walk: whatever box a ray really enters is among the leaves either tree reaches, and the trees do cull
    most, reached = check_walks(t, lo, hi)
    assert most < max(64, 0.2 * len(lo)) or len(lo) < 1000
    assert reached > 0 or len(lo) < 3


def test_host_bvh_rejects_what_the_reference_panics_on(rt):
    api = rt.api
    with pytest.raises(api.Rt1wError):  # bvh.rs:61: "No objects in bvh_node constructor."
        api.build_bvh_host(np.zeros((0, 3)), np.zeros((0, 3)))
    with pytest.raises(api.Rt1wError):  # bvh.rs:65-67: "No bounding box in bvh_node constructor."
        api.build_bvh_host(np.array([[0.0, 0.0, -np.inf]]), np.array([[1.0, 1.0, np.inf]]))
