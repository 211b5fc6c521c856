"""The device BVH builder of scene commit (csrc/lbvh.cu, with the box padding of csrc/bvh.cpp that api.cu: lbvh_build applies
first) restated in numpy, vectorised over nodes, so that its output can be compared with the device's bit for bit.

Every step is integer arithmetic, an f32 operation numpy rounds the same way, or an f32 min / max:
  * conservative_box: per axis pad = 1e-5 ext + 1e-5 + 1e-6 reach in f64 (ext = max(hi - lo, |lo|, |hi|), reach = the
    largest coordinate of all boxes), lo - pad and hi + pad rounded to f32, then one f32 step outward (nextafter);
  * the centroid box on the host: c = 0.5f (lo + hi) in f32, its per-axis min / max, inv = 1 / (max - min) in f32, or 0
    on an axis without extent;
  * k_morton: ((c - min) * inv) * (2^21 - 1) in f32, clamped to [0, 2^21 - 1] and truncated, three 21-bit values
    interleaved into 63 bits (x highest).  The one place FMA contraction could act, c - min, is exact there because the
    product 0.5 (lo + hi) is exact (denormal coordinates excepted);
  * cub::DeviceRadixSort::SortPairs on (key, input index): a stable sort;
  * k_topology (Karras 2012) with the same tie-break: delta(i, j) = 64 + clz32(i ^ j) for equal keys;
  * k_fit: every interior box the f32 min / max of its leaves' boxes (min and max are exact, so the order of the reduction
    does not matter), the height of the root;
  * k_emit: node 0 the root, node 1 zeros, the children of interior node i at 2 + 2 i and 3 + 2 i; a leaf has
    left_first = its sorted position and count = 1, an interior node c has left_first = 2 + 2 c and count = 0."""
import numpy as np

NODE_DTYPE = np.dtype([("min", np.float32, 3), ("left_first", np.uint32), ("max", np.float32, 3), ("count", np.uint32)])  # bvh.h: BvhNode32
F32 = np.float32
QMAX = F32(2097151.0)  # 2^21 - 1


def conservative_boxes(lo, hi, outward=True):
    """bvh.cpp: traversal_pad + conservative_box over every box, as api.cu: lbvh_build pads them. -> (n, 6) float32."""
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    reach = max(np.abs(lo).max(), np.abs(hi).max())
    ext = np.maximum(hi - lo, np.maximum(np.abs(lo), np.abs(hi)))
    pad = 1e-5 * ext + 1e-5 + 1e-6 * reach
    l, h = (lo - pad).astype(F32), (hi + pad).astype(F32)
    if not outward:  # the mutation of build(outward=False)
        return np.concatenate([l, h], axis=1)
    return np.concatenate([np.nextafter(l, F32(-np.inf)), np.nextafter(h, F32(np.inf))], axis=1)


def _spread21(v):
    x = v.astype(np.uint64) & np.uint64(0x1FFFFF)
    for sh, m in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3), (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(sh))) & np.uint64(m)
    return x


def morton_keys(boxes):
    """The host's centroid box and k_morton's 63-bit keys of the padded f32 boxes."""
    c = F32(0.5) * (boxes[:, :3] + boxes[:, 3:])
    clo, chi = c.min(axis=0), c.max(axis=0)
    ext = chi - clo
    inv = np.where(chi > clo, F32(1.0) / np.where(chi > clo, ext, F32(1.0)), F32(0.0)).astype(F32)
    q = np.minimum(np.maximum(((c - clo) * inv) * QMAX, F32(0.0)), QMAX).astype(np.uint32)
    return _spread21(q[:, 0]) << np.uint64(2) | _spread21(q[:, 1]) << np.uint64(1) | _spread21(q[:, 2])


def _bit_length(x):
    """Bit length of every uint64 (frexp is exact on 32-bit halves)."""
    hi, lo = (x >> np.uint64(32)).astype(np.float64), (x & np.uint64(0xFFFFFFFF)).astype(np.float64)
    return np.where(hi > 0, 32 + np.frexp(hi)[1], np.frexp(lo)[1]).astype(np.int64)


def _delta(keys, i, j):
    """lbvh.cu: delta, elementwise: -1 outside [0, n), the common prefix of the keys, 64 + clz32(i ^ j) for equal keys."""
    n = len(keys)
    ok = (j >= 0) & (j < n)
    jj = np.where(ok, j, 0)
    a, b = keys[i], keys[jj]
    same = 64 + 32 - _bit_length((i ^ jj).astype(np.uint64) & np.uint64(0xFFFFFFFF))
    diff = 64 - _bit_length(a ^ b)
    out = np.where(a == b, same, diff)
    return np.where(ok, out, -1)


def topology(keys):
    """k_topology over sorted keys: per interior node i its two children (index, is_leaf) and its leaf range."""
    n = len(keys)
    i = np.arange(n - 1, dtype=np.int64)
    dl = lambda j: _delta(keys, i, j)
    d = np.where(dl(i + 1) - dl(i - 1) >= 0, 1, -1)
    dmin = dl(i - d)
    lmax = np.full(n - 1, 2, np.int64)
    grow = dl(i + lmax * d) > dmin
    while grow.any():
        lmax = np.where(grow, 2 * lmax, lmax)
        grow &= dl(i + lmax * d) > dmin
    l, t = np.zeros(n - 1, np.int64), lmax // 2
    while (t >= 1).any():
        l += np.where((t >= 1) & (dl(i + (l + t) * d) > dmin), t, 0)
        t //= 2
    j = i + l * d
    dnode = dl(j)
    s, t, go = np.zeros(n - 1, np.int64), l.copy(), np.ones(n - 1, bool)
    while go.any():  # do { t = (t + 1) / 2; ... } while (t > 1)
        t = np.where(go, (t + 1) // 2, t)
        s += np.where(go & (dl(i + (s + t) * d) > dnode), t, 0)
        go &= t > 1
    gamma = i + s * d + np.minimum(d, 0)
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    child = np.stack([gamma, gamma + 1], axis=1)
    leaf = np.stack([lo == gamma, hi == gamma + 1], axis=1)
    return child, leaf, lo, hi


def _range_reduce(ufunc, a, lo, hi):
    """ufunc over a[lo[k] : hi[k] + 1] for every k (queries sorted by lo so that reduceat's gaps stay short)."""
    srt = np.argsort(lo, kind="stable")
    idx = np.stack([lo[srt], hi[srt] + 1], axis=1).ravel()
    padded = np.concatenate([a, a[:1]])  # hi + 1 may be n
    out = np.empty((len(lo), a.shape[1]), a.dtype)
    out[srt] = ufunc.reduceat(padded, idx, axis=0)[::2]
    return out


def build(lo, hi, outward=True):
    """The device builder's output for boxes (n, 3) f64 lo / hi: dict(nodes (2 n NODE_DTYPE), prim_order (uint32), depth,
    keys (sorted)).  outward=False is a deliberate one-line mutation that the exactness tests must catch: boxes without
    the final f32 step outward, one ulp too small - the kind of error that only loses grazing hits."""
    boxes = conservative_boxes(lo, hi, outward)
    n = len(boxes)
    assert n >= 2
    keys = morton_keys(boxes)
    order = np.argsort(keys, kind="stable").astype(np.uint32)
    skeys = keys[order]
    child, leaf, rlo, rhi = topology(skeys)
    sb = boxes[order]
    ilo = _range_reduce(np.minimum, sb[:, :3], rlo, rhi)
    ihi = _range_reduce(np.maximum, sb[:, 3:], rlo, rhi)
    # heights: the depth of every interior node by pointer jumping, the root's height = the deepest leaf's depth
    parent = np.zeros(n - 1, np.int64)
    for side in (0, 1):
        m = ~leaf[:, side]
        parent[child[m, side]] = np.flatnonzero(m)
    dist = np.ones(n - 1, np.int64)
    dist[0] = 0
    anc = parent.copy()
    for _ in range(8):  # 2^8 levels: the tie-break caps the height at 63 + 32
        if not (anc != 0).any():
            break
        dist, anc = dist + dist[anc], anc[anc]
    assert not (anc != 0).any(), "the parent links do not reach the root"
    depth = int(np.where(leaf, dist[:, None] + 1, 0).max())
    nodes = np.zeros(2 * n, NODE_DTYPE)
    nodes[0]["min"], nodes[0]["max"], nodes[0]["left_first"] = ilo[0], ihi[0], 2
    for side in (0, 1):
        at = 2 + 2 * np.arange(n - 1) + side
        c, lf = child[:, side], leaf[:, side]
        nodes["min"][at] = np.where(lf[:, None], sb[c, :3], ilo[np.where(lf, 0, c)])
        nodes["max"][at] = np.where(lf[:, None], sb[c, 3:], ihi[np.where(lf, 0, c)])
        nodes["left_first"][at] = np.where(lf, c, 2 + 2 * c)
        nodes["count"][at] = lf
    return dict(nodes=nodes, prim_order=order, depth=depth, keys=skeys)



# --------------------------------------------------------------------------- inputs of the tests (f64 lo, hi boxes)
def random_boxes(n, seed, offset=0.0, size_range=(0.05, 3.0), log_sizes=False):
    rng = np.random.Generator(np.random.Philox(seed))
    c = offset + rng.uniform(-100, 100, (n, 3))
    r = np.exp(rng.uniform(np.log(size_range[0]), np.log(size_range[1]), (n, 3))) if log_sizes else rng.uniform(*size_range, (n, 3))
    return c - r, c + r


def scene_boxes(api, name, **kw):
    """The world boxes of a shipped scene's lowered primitives (api.lower_prims, read straight from the ctypes buffer: a
    million-primitive scene in a fraction of a second), the finite ones."""
    import ctypes as C

    hs = api.HostScene(name, seed=1, **kw)
    lib, n = api.load_library(), C.c_int32(0)
    dp = C.pointer(hs.desc) if not isinstance(hs.desc, C.POINTER(api.SceneDesc)) else hs.desc
    assert lib.rt1w_lower_prims(dp, None, 0, C.byref(n)) == api.OK
    buf = (api.FlatPrim * n.value)()
    assert lib.rt1w_lower_prims(dp, buf, n.value, C.byref(n)) == api.OK
    dt = np.dtype(dict(names=["lo", "hi"], formats=[(np.float64, 3), (np.float64, 3)], itemsize=C.sizeof(api.FlatPrim),
                       offsets=[api.FlatPrim.bbox_min.offset, api.FlatPrim.bbox_max.offset]))
    a = np.frombuffer(buf, dtype=dt)
    ok = np.isfinite(a["lo"]).all(1) & np.isfinite(a["hi"]).all(1)
    return a["lo"][ok].copy(), a["hi"][ok].copy()


def chain(corner=True, origin_dups=0, deep_radii=False, first_m=0):
    """Spheres (centres, radii) at quantised single-bit positions: one at the origin, one at (2^m + 0.5) e_axis for
    m = first_m..20 on each axis, the corner (2^21 - 1) (1, 1, 1) if corner, origin_dups more at the origin.  Every Morton
    key is one bit on top of the keys before it, so the LBVH is a chain: 63 levels with the corner sphere, 60 without, 70
    with 64 duplicates at the origin.  The 8-wide collapse takes seven chain levels per node, but only three levels of the
    balanced subtree that duplicates form: from m = 4 with 3000 duplicates the LBVH has 60 levels and its collapse 11.  deep_radii: radii 2^m + 1 + (3 m + axis + 1) / 256 (all distinct, so no two spheres share
    an extreme point) instead of 0.25 and 0.1 at the origin: every box but the origin sphere's contains the ball of radius
    0.5 around the origin, so a ray from there enters both children of every interior node above that sphere."""
    c, r = [(0.0, 0.0, 0.0)], [0.1 if deep_radii else 0.25]
    if corner:
        c.append((2097151.0,) * 3), r.append(0.25)
    for m in range(first_m, 21):
        for ax in range(3):
            p = [0.0, 0.0, 0.0]
            p[ax] = 2.0 ** m + 0.5
            c.append(tuple(p)), r.append(2.0 ** m + 1.0 + (3 * m + ax + 1) / 256.0 if deep_radii else 0.25)
    c += [(0.0, 0.0, 0.0)] * origin_dups
    r += [0.25] * origin_dups
    return np.array(c), np.array(r)


def _spheres(c, r):
    return c - r[:, None], c + r[:, None]


def _identical(n=1000):
    """Boxes of many sizes about the origin: padding and rounding are symmetric there, so every f32 centroid is 0."""
    rng = np.random.Generator(np.random.Philox(3))
    r = rng.uniform(0.1, 2.0, (n, 3))
    return -r, r


def _duplicate_runs():
    rng = np.random.Generator(np.random.Philox(4))
    c = rng.uniform(-50, 50, (300, 3))
    c = np.concatenate([np.repeat(c, rng.integers(1, 9, 300), axis=0), rng.uniform(-50, 50, (500, 3))])
    c = c[rng.permutation(len(c))]
    r = rng.uniform(0.1, 1.0, (len(c), 1))
    return c - r, c + r


def _flat(axes):
    lo, hi = random_boxes(3000, 5)
    for ax in axes:  # symmetric boxes about one coordinate: all centroids on the plane / line
        h = np.abs(hi[:, ax] - lo[:, ax]) / 2
        lo[:, ax], hi[:, ax] = 3.0 - h, 3.0 + h
    return lo, hi


def _extremes():
    rng = np.random.Generator(np.random.Philox(6))
    c = rng.uniform(-10, 10, (2000, 3))
    c[:1000] = np.where(rng.random((1000, 3)) < 0.5, -10.0, 10.0)  # corners: every coordinate at its axis' min or max
    c[1000:1200, 0], c[1200:1400, 1] = -10.0, 10.0
    r = rng.uniform(0.01, 0.5, (2000, 1))
    return c - r, c + r


# name -> f(api) -> (lo, hi)
INPUTS = {
    **{f"n{n}": (lambda n: lambda api: random_boxes(n, 100 + n))(n) for n in (2, 3, 4, 255, 256, 257, 4097)},
    "random_scene": lambda api: scene_boxes(api, "random_scene"),
    "final_scene": lambda api: scene_boxes(api, "final_scene"),
    "stress_200k": lambda api: scene_boxes(api, "stress", stress_spheres=200_000),
    "identical_1000": lambda api: _identical(),
    "duplicate_runs": lambda api: _duplicate_runs(),
    "plane": lambda api: _flat([2]),
    "line": lambda api: _flat([1, 2]),
    "offset_1e6": lambda api: random_boxes(3000, 7, offset=1e6),
    "sizes_1e6": lambda api: random_boxes(3000, 8, size_range=(1e-3, 1e3), log_sizes=True),
    "extremes": lambda api: _extremes(),
    "chain_65": lambda api: _spheres(*chain()),
    "chain_129": lambda api: _spheres(*chain(origin_dups=64)),
    "chain_64": lambda api: _spheres(*chain(corner=False)),
    "chain_64_deep": lambda api: _spheres(*chain(corner=False, deep_radii=True)),
    "chain_wide": lambda api: _spheres(*chain(corner=False, origin_dups=3000, first_m=4)),
}
# the heights these inputs must give
DEPTHS = {"identical_1000": 10, "chain_65": 63, "chain_129": 70, "chain_64": 60, "chain_64_deep": 60, "chain_wide": 60}
