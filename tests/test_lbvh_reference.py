"""The numpy restatement of the device BVH builder (tests/lbvh_reference.py) on the CPU, so that the reference the GPU tests
hold lbvh.cu to is pinned without a GPU:
  * its trees pass the structural and conservativeness checks of the host SAH tree (common.check_binary) on every input of
    the GPU exactness test, with the heights the inputs are built to have (one shared centroid: ceil(log2 n); the chains);
  * its vectorised Karras topology equals a plain recursive binary radix tree over the keys extended by their sorted index
    (the tie-break of lbvh.cu: delta), node for node."""
import numpy as np
import pytest

import lbvh_reference as ref
from common import check_binary

MAX_HEIGHT = 63 + 32  # 63 key bits + 32 index bits: the most levels the tie-broken radix tree can have


@pytest.mark.parametrize("name", list(ref.INPUTS))
def test_reference_trees_pass_the_tree_checks(rt, name):
    lo, hi = ref.INPUTS[name](rt.api)
    t = ref.build(lo, hi)
    assert len(t["nodes"]) == 2 * len(lo)
    assert t["nodes"][1].tobytes() == bytes(32), "node 1 is padding, all zeros"
    n_nodes = check_binary(t, lo, hi, max_depth_allowed=62 if t["depth"] <= 62 else MAX_HEIGHT)
    assert n_nodes == 2 * len(lo) - 1
    if name in ref.DEPTHS:
        assert t["depth"] == ref.DEPTHS[name]


def _radix_tree(keys):
    """{(first, last): split} of the binary radix tree over sorted 63-bit keys extended by 32 index bits, by recursion."""
    ext = [(int(k) << 32) | i for i, k in enumerate(keys)]
    out, todo = {}, [(0, len(keys) - 1)]
    while todo:
        a, b = todo.pop()
        if a == b:
            continue
        prefix = 96 - (ext[a] ^ ext[b]).bit_length()
        g = max(x for x in range(a, b) if 96 - (ext[a] ^ ext[x]).bit_length() > prefix)  # the last key that shares more with a
        out[(a, b)] = g
        todo += [(a, g), (g + 1, b)]
    return out


@pytest.mark.parametrize("name", ["n2", "n3", "n257", "identical_1000", "duplicate_runs", "chain_65", "chain_129", "extremes"])
def test_topology_is_the_binary_radix_tree(rt, name):
    lo, hi = ref.INPUTS[name](rt.api)
    keys = np.sort(ref.morton_keys(ref.conservative_boxes(lo, hi)), kind="stable")
    child, leaf, first, last = ref.topology(keys)
    got = {(int(a), int(b)): int(g) for a, b, g in zip(first, last, child[:, 0])}
    assert got == _radix_tree(keys)
    assert (leaf[:, 0] == (child[:, 0] == first)).all() and (leaf[:, 1] == (child[:, 1] == last)).all()
