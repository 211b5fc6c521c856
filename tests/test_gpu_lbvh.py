"""The device-side BVH builder (lbvh.cu): bit for bit against its numpy restatement (tests/lbvh_reference.py), the commit's
fall-backs for trees too deep for the traversal stacks, traversal at the depth limit, and against the host SAH builder
(same closest hits, same renders).

Exactness: rt1w_build_bvh_device (the commit's own padding, build and copy back) against lbvh_reference.build on every
input of lbvh_reference.INPUTS - sizes around the 256-thread blocks, the boxes of random_scene, final_scene and the stress
scene with 2 * 10^5 spheres, 1000 boxes with one centroid, runs of duplicates, centroids on a plane and on a line, a cloud
10^6 from the origin, sizes 10^6 apart, centroids at the per-axis extremes and the chains - and once on the 10^6-sphere
stress scene: all 2 n nodes as raw bytes, the primitive order and the height.  The trees also pass the structure,
conservativeness and reference-walk checks of the host SAH tree (common.py; the 10^6 tree is only compared).  Builds
repeat bit for bit, and on a second GPU give the same bytes.

Fall-backs and depth limit (lbvh_reference.chain: spheres at single-bit Morton positions, so the LBVH is a chain):
  * 65 and 129 spheres (LBVH heights 63 and 70): scene commit falls back to the SAH tree - its depth and leaf table, and
    closest hits that match the oracle;
  * 64 spheres (height 60, the deepest chain the commit keeps) collapse into 8 wide levels: seven chain levels per wide
    node.  A chain from m = 4 over 3000 coincident spheres (height 60) collapses into 11, deeper than kWideMaxDepth, so
    the scene keeps the binary walk, and a render asked for the wide tree equals the binary render bit for bit;
  * the same 64 spheres with radii just above 2^m + 1: every box contains a neighbourhood of the origin, so a ray from there
    enters both children of every interior node and pushes one stack entry per level, far into the local-memory overflow
    (the kernels' push rule replayed in numpy proves the depth); closest hits against the oracle, 1-spp renders of every
    binary-tree kernel against the host replay of each path, and the feature buffers against the camera-ray and trace hooks."""
import os

import numpy as np
import pytest

import lbvh_reference as ref
from common import check_binary, check_identical_render, check_trace_parity, check_walks, check_wide, make_ray_set, pixel_seeds

pytestmark = pytest.mark.gpu


def _scene(api, ctx, desc, builder):
    old = os.environ.get("RT1W_BVH_BUILDER")
    os.environ["RT1W_BVH_BUILDER"] = builder
    try:
        return api.Scene(ctx, desc)
    finally:
        if old is None:
            del os.environ["RT1W_BVH_BUILDER"]
        else:
            os.environ["RT1W_BVH_BUILDER"] = old


@pytest.mark.parametrize("name,extent", [("random_scene", 30.0), ("final_scene", None)])
def test_lbvh_finds_the_same_hits(rt, oracle, gpu_ctx, name, extent):
    api = rt.api
    hs = api.HostScene(name, seed=1)
    osc = oracle.OracleScene(hs.desc)
    sah, lbvh = _scene(api, gpu_ctx, hs.desc, "sah"), _scene(api, gpu_ctx, hs.desc, "lbvh")
    assert lbvh.info().n_bvh_nodes >= 2 and lbvh.info().bvh_depth >= 1
    rays = make_ray_set(api, hs, osc, sah.prims(), 1 << 16, max_extent=extent)
    pa, ta, na, fa, _ = sah.trace_closest(rays, seed=7)
    pb, tb, nb, fb, _ = lbvh.trace_closest(rays, seed=7)
    same = pa == pb
    # two leaves at the same distance (a box lying on the floor, coincident sides) may swap with the traversal order
    assert same.mean() >= 0.999
    hit = same & (pa >= 0)
    assert np.array_equal(ta[hit], tb[hit]) and np.array_equal(na[hit], nb[hit]) and np.array_equal(fa[hit], fb[hit])
    differ = ~same
    assert np.allclose(ta[differ], tb[differ], rtol=1e-6)
    sah.close(), lbvh.close()


def test_lbvh_render_agrees(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    sah, lbvh = _scene(api, gpu_ctx, hs.desc, "sah"), _scene(api, gpu_ctx, hs.desc, "lbvh")
    cam = hs.camera()
    for flags in (api.FLAG_BVH_LOCKSTEP, api.FLAG_BVH_PERSISTENT):
        a, _, sa = sah.render(cam, hs.params(width=96, spp=16, seed=5, flags=flags))
        b, _, sb = lbvh.render(cam, hs.params(width=96, spp=16, seed=5, flags=flags))
        assert abs(int(sa.rays) - int(sb.rays)) <= 1e-4 * sa.rays  # ties at equal distance may end a path elsewhere
        assert abs(np.nan_to_num(a).mean() - np.nan_to_num(b).mean()) <= 0.01 * np.nan_to_num(a).mean()
        close = np.isclose(a, b, rtol=1e-3, atol=1e-3) | ~np.isfinite(a) | ~np.isfinite(b)
        assert close.mean() >= 0.999
    sah.close(), lbvh.close()


# --------------------------------------------------------------------------- exactness against the numpy restatement
def _same_tree(got, want, label):
    """All 2 n nodes as raw bytes, the primitive order and the height; on failure the first differing nodes, field by field."""
    assert got["depth"] == want["depth"], f"{label}: height {got['depth']}, reference {want['depth']}"
    assert np.array_equal(got["prim_order"], want["prim_order"]), \
        f"{label}: primitive order differs first at sorted position {np.flatnonzero(got['prim_order'] != want['prim_order'])[:5]}"
    g, w = got["nodes"], want["nodes"]
    assert g.shape == w.shape, f"{label}: {len(g)} nodes, reference {len(w)}"
    bad = np.flatnonzero((g.view(np.uint8).reshape(len(g), -1) != w.view(np.uint8).reshape(len(w), -1)).any(1))
    assert bad.size == 0, f"{label}: {bad.size} of {len(g)} nodes differ; first ones:\n" + "\n".join(
        f"  node {k}: device {g[k]} reference {w[k]}" for k in bad[:5])


DEEP = {"chain_65", "chain_129"}  # heights above 62: trees the commit refuses


@pytest.mark.parametrize("name", list(ref.INPUTS))
def test_device_builder_is_the_reference(rt, gpu_ctx, name):
    api = rt.api
    lo, hi = ref.INPUTS[name](api)
    got = api.build_bvh_device(gpu_ctx, lo, hi)
    _same_tree(got, ref.build(lo, hi), name)
    if name in ref.DEPTHS:
        assert got["depth"] == ref.DEPTHS[name]
    assert check_binary(got, lo, hi, max_depth_allowed=95 if name in DEEP else 62) == 2 * len(lo) - 1
    too_wide = name in ("chain_129", "chain_wide")  # collapses deeper than the wide walk's stack (kWideMaxDepth = 10)
    check_wide(got, lo, hi, max_wide_depth=got["wide_depth"] if too_wide else 10)
    assert (got["wide_depth"] > 10) == too_wide
    check_walks(got, lo, hi)


def test_a_mutated_reference_is_caught(rt, gpu_ctx):
    """The exactness bar has teeth: the reference without the final f32 step outward of conservative_box (one line: node
    boxes one ulp too small, which only grazing rays would notice) differs from the device."""
    api = rt.api
    lo, hi = ref.INPUTS["final_scene"](api)
    got = api.build_bvh_device(gpu_ctx, lo, hi)
    _same_tree(got, ref.build(lo, hi), "final_scene")
    with pytest.raises(AssertionError, match="nodes differ"):
        _same_tree(got, ref.build(lo, hi, outward=False), "final_scene, mutated reference")


def _n_gpus():
    import torch

    return torch.cuda.device_count()


def test_million_sphere_tree_is_the_reference_and_repeats(rt, gpu_ctx):
    api = rt.api
    lo, hi = ref.scene_boxes(api, "stress", stress_spheres=1_000_000)
    a = api.build_bvh_device(gpu_ctx, lo, hi)
    _same_tree(a, ref.build(lo, hi), "stress 10^6")
    _same_tree(api.build_bvh_device(gpu_ctx, lo, hi), a, "stress 10^6, second build")
    assert np.array_equal(api.build_bvh_device(gpu_ctx, lo, hi)["wide_nodes"].view(np.uint8), a["wide_nodes"].view(np.uint8))
    if _n_gpus() >= 2:
        ctx1 = api.Context(1)
        try:
            _same_tree(api.build_bvh_device(ctx1, lo, hi), a, "stress 10^6 on device 1")
        finally:
            ctx1.close()


def test_device_builder_rejects_what_the_host_builder_rejects(rt, gpu_ctx):
    api = rt.api
    for lo, hi in ((np.zeros((0, 3)), np.zeros((0, 3))), (np.zeros((1, 3)), np.ones((1, 3))),
                   (np.array([[0.0, 0.0, 0.0], [0.0, 0.0, -np.inf]]), np.array([[1.0, 1.0, 1.0], [1.0, 1.0, np.inf]])),
                   (np.array([[0.0, 0.0, 0.0], [np.nan, 0.0, 0.0]]), np.ones((2, 3)))):
        with pytest.raises(api.Rt1wError) as e:
            api.build_bvh_device(gpu_ctx, lo, hi)
        assert e.value.status == api.ERR_INVALID


# --------------------------------------------------------------------------- scene commit: fall-backs and the depth limit
class _Chain:
    """A chain scene (lbvh_reference.chain) as a scene description, with what make_ray_set and the renders need."""

    class _Settings:
        pass

    def __init__(self, api, centres, radii, lights=()):
        b = api.DescBuilder()
        greys = [b.lambertian(b.solid(*c)) for c in ((0.7, 0.7, 0.7), (0.8, 0.3, 0.2), (0.2, 0.6, 0.3), (0.3, 0.4, 0.8))]
        lamp = b.diffuse_light(b.solid(1.5, 1.4, 1.2))
        kids = []
        for k, (c, r) in enumerate(zip(centres, radii)):
            if k in lights:  # lit from the inside: the camera sits inside these spheres
                kids.append(b.flip_face(b.sphere(tuple(c), float(r), lamp)))
            else:
                kids.append(b.sphere(tuple(c), float(r), greys[k % 4]))
        b.set_world(b.bvh(kids))
        self.api, self.b, self.desc = api, b, b.desc()
        self.centres, self.radii = centres, radii
        self.look_from, self.background = (-6.0, 5.0, -7.0), (0.6, 0.7, 0.9)
        self.settings = self._Settings()
        self.settings.look_at = (2.0, 1.0, 1.0)

    def camera(self, aspect=1.0):
        return self.api.camera_new(self.look_from, self.settings.look_at, (0.0, 1.0, 0.0), 60.0, aspect, 0.0, 10.0, 0.0, 1.0)

    def params(self, width, s=0, flags=0, max_depth=50, seed=0):
        p = self.api.RenderParams()
        p.width = p.height = width
        p.sample_begin, p.sample_end, p.max_depth, p.flags, p.seed = s, s + 1, max_depth, flags, seed
        p.background[:] = list(self.background)
        return p


def _commit(api, ctx, desc, builder, monkeypatch):
    with monkeypatch.context() as m:
        m.setenv("RT1W_BVH_BUILDER", builder)
        return api.Scene(ctx, desc)


def _aimed_rays(api, centres, radii, n, seed):
    """Rays at points inside random spheres from 1 - 1000 units away: most of them hit something, and none from so far
    that a 0.25 sphere's f64 discriminant cancels to its last bits."""
    rng = np.random.Generator(np.random.Philox(seed))
    k = rng.choice(np.flatnonzero(np.abs(centres).sum(1) > 0), n)  # (not the origin: duplicates there are exact ties)
    target = centres[k] + 0.8 * radii[k, None] * rng.uniform(-1.0, 1.0, (n, 3)) / np.sqrt(3.0)
    u = rng.normal(size=(n, 3))
    origin = target + u / np.linalg.norm(u, axis=1, keepdims=True) * np.exp(rng.uniform(0.0, np.log(1000.0), (n, 1)))
    rays = np.zeros(n, dtype=api.RAY_DTYPE)
    rays["origin"], rays["direction"] = origin, target - origin
    rays["time"] = rng.random(n)
    return rays


def _sphere_ties(rays, centres, radii):
    """Rays whose closest sphere hit (world.hit(ray, 0.001, inf), every sphere solved in f64 from the f32 ray) is not robust:
    another sphere within 1e-6 relative of it, or a sphere grazed no farther away (a discriminant within 1e-12 of the terms
    it cancels: 10^4 times the f64 rounding of either solver).
    The oracle's own screen perturbs ray origins by 1e-9 of the scene's extent, 4e-3 here, which moves every hit on
    the small spheres near the origin; these scenes hold spheres only, so the screen is computed exactly instead."""
    o = rays["origin"].astype(np.float64)[:, None, :] - centres[None]
    d = rays["direction"].astype(np.float64)[:, None, :]
    a, hb = (d * d).sum(-1), (o * d).sum(-1)
    cc = (o * o).sum(-1) - radii[None] ** 2
    disc = hb * hb - a * cc
    sq = np.sqrt(np.maximum(disc, 0.0))
    t0, t1 = (-hb - sq) / a, (-hb + sq) / a
    t = np.where(disc < 0, np.inf, np.where(t0 >= 0.001, t0, np.where(t1 >= 0.001, t1, np.inf)))
    ts = np.sort(t, axis=1)
    best = ts[:, 0]
    with np.errstate(invalid="ignore"):  # inf - inf: rays that hit one sphere or none
        tie = np.isfinite(best) & (ts[:, 1] - best <= 1e-6 * best)
    graze = (np.abs(disc) <= 1e-12 * (hb * hb + np.abs(a * cc))) & (-hb / a <= best[:, None] * (1 + 1e-6) + 1e-9)
    return tie | graze.any(1) | (np.abs(best - 0.001) < 1e-9)


def _trace_parity(gsc, osc, rays, centres, radii, label):
    """check_trace_parity's bars (primitive ids exact, t and normals within 1e-5, front faces, (u, v)) against the oracle, on
    every ray _sphere_ties does not screen out."""
    op, ot, on, off, ouv, _ = osc.trace_closest(rays, seed=0x5EED)
    amb = _sphere_ties(rays, centres, radii).astype(np.uint8)
    return check_trace_parity(gsc, osc, rays, label=label, cache={"trace": (op, ot, on, off, ouv, amb)})


@pytest.mark.parametrize("dups", [0, 64], ids=["chain_65", "chain_129"])
def test_too_deep_lbvh_falls_back_to_sah(rt, oracle, gpu_ctx, monkeypatch, dups):
    api = rt.api
    c, r = ref.chain(origin_dups=dups)
    sc = _Chain(api, c, r)
    assert api.build_bvh_device(gpu_ctx, c - r[:, None], c + r[:, None])["depth"] == (63 if dups == 0 else 70)
    lbvh, sah = _commit(api, gpu_ctx, sc.desc, "lbvh", monkeypatch), _commit(api, gpu_ctx, sc.desc, "sah", monkeypatch)
    li, si = lbvh.info(), sah.info()
    print(f"[lbvh] chain of {len(c)} spheres: LBVH height > 62, committed depth {li.bvh_depth} (SAH {si.bvh_depth})")
    assert li.bvh_depth == si.bvh_depth <= 62 and li.n_bvh_nodes == si.n_bvh_nodes
    assert np.array_equal(lbvh.leaf_prims(), sah.leaf_prims())
    osc = oracle.OracleScene(sc.desc)
    _trace_parity(lbvh, osc, _aimed_rays(api, c, r, 1 << 15, 3), c, r, f"chain of {len(c)}, LBVH fell back")
    lbvh.close(), sah.close()


def test_deepest_accepted_lbvh_keeps_the_binary_walk(rt, gpu_ctx, monkeypatch):
    """A tree the commit keeps (60 levels) whose 8-wide collapse is deeper than the wide walk's stack (11 levels: a chain
    over 3000 coincident spheres): the scene keeps the binary walk, and a render asked for the wide tree is the binary one."""
    api = rt.api
    c, r = ref.chain(corner=False, origin_dups=3000, first_m=4)
    sc = _Chain(api, c, r)
    t = api.build_bvh_device(gpu_ctx, c - r[:, None], c + r[:, None])
    assert t["depth"] == 60 and t["wide_depth"] > 10
    gsc = _commit(api, gpu_ctx, sc.desc, "lbvh", monkeypatch)
    info = gsc.info()
    assert info.bvh_depth == 60 and info.wide_depth == t["wide_depth"] and info.wide_default == 0
    cam = sc.camera()
    for s in (0, 7):
        a = gsc.render(cam, sc.params(64, s, api.FLAG_BVH_WIDE))
        b = gsc.render(cam, sc.params(64, s, api.FLAG_BVH_BINARY))
        check_identical_render(a, b, f"chain over 3000 coincident spheres, sample {s}: wide flag vs binary", 1, s)
    gsc.close()


def _deep_scene(api):
    c, r = ref.chain(corner=False, deep_radii=True)
    lights = [k for k in range(1, len(c)) if (k - 1) % 3 == 1]  # the spheres on the y axis
    sc = _Chain(api, c, r, lights=lights)
    sc.look_from, sc.settings.look_at = (0.2, 0.25, 0.3), (3.0, 0.5, 1.0)  # inside every sphere but the one at the origin
    return sc


def _ball_rays(api, n, seed):
    """Rays from 0.15 - 0.45 around the origin (outside its 0.1 sphere, inside every other box) in all directions."""
    rng = np.random.Generator(np.random.Philox(seed))
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    rays = np.zeros(n, dtype=api.RAY_DTYPE)
    rays["origin"] = u * rng.uniform(0.15, 0.45, (n, 1))
    rays["direction"] = rng.normal(size=(n, 3))
    rays["time"] = rng.random(n)
    return rays


def _first_descent_stack(nodes, rays):
    """The traversal stack of kernels.cuh (trav_step_interior) on each ray's first descent, replayed in numpy: both children
    tested with slab's FMA form on the f32 ray, the nearer entry distance first (tl <= tr takes the left child), the other
    pushed.  No leaf has been reached yet, so nothing is culled by a hit: these are the exact stack heights the kernels
    reach before their first primitive test."""
    f = np.float32
    o, d = rays["origin"].astype(f), rays["direction"].astype(f)
    inv = (f(1.0) / np.copysign(np.maximum(np.abs(d), f(1e-18)), d)).astype(f)  # rcp_capped (rcp.approx: within an ulp)
    oo = (-o * inv).astype(f)

    def entry(k):
        lo, hi = nodes["min"][k].astype(np.float64), nodes["max"][k].astype(np.float64)
        a = (lo * inv + oo).astype(f)
        b = (hi * inv + oo).astype(f)
        tn = np.maximum(np.minimum(a, b).max(1), f(0.0))
        return tn, tn <= np.maximum(a, b).min(1)

    ref_ = np.zeros(len(rays), np.int64)  # node index (0 = root; assumed entered: the rays start inside its box)
    sp = np.zeros(len(rays), np.int64)
    live = nodes["count"][0] == 0
    live = np.full(len(rays), live)
    while live.any():
        left = nodes["left_first"][ref_].astype(np.int64)
        tl, hl = entry(left)
        tr, hr = entry(left + 1)
        both = live & hl & hr
        sp += both
        nxt = np.where(hl & (~hr | (tl <= tr)), left, left + 1)
        live &= hl | hr
        ref_ = np.where(live, nxt, ref_)
        live &= nodes["count"][ref_] == 0
    return sp


def test_traversal_at_the_depth_limit(rt, oracle, gpu_ctx, monkeypatch):
    """Closest hits, every path of 1-spp renders and the feature buffers on a scene whose rays fill the binary traversal
    stack to 60 entries: 16 in shared memory, 44 in the local-memory overflow."""
    from test_gpu_path_replay import MAX_ALL, MAX_UNFLAGGED, match

    api = rt.api
    sc = _deep_scene(api)
    c, r = sc.centres, sc.radii
    t = api.build_bvh_device(gpu_ctx, c - r[:, None], c + r[:, None])
    assert t["depth"] == 60
    ball = _ball_rays(api, 1 << 14, 5)
    stack = _first_descent_stack(t["nodes"], ball)
    print(f"[lbvh] depth-limit scene: tree height {t['depth']}, first-descent stack up to {stack.max()} entries "
          f"(median {int(np.median(stack))})")
    assert stack.max() >= 48 and np.median(stack) >= 48, "the ray set does not reach deep into the stack overflow"
    gsc = _commit(api, gpu_ctx, sc.desc, "lbvh", monkeypatch)
    info = gsc.info()
    assert info.bvh_depth == 60 and info.wide_default == 0 and info.n_global_prims == 0
    osc = oracle.OracleScene(sc.desc)
    _trace_parity(gsc, osc, ball, c, r, "depth-limit scene, rays from the origin's neighbourhood")
    _trace_parity(gsc, osc, make_ray_set(api, sc, osc, gsc.prims(), 1 << 15, max_extent=8.0), c, r, "depth-limit scene, ray mix")
    # every path of 1-spp renders against its host replay (test_gpu_path_replay.py's bars), on every binary-tree kernel
    cam = sc.camera()
    leaf = oracle.replay_leaf_map(gsc.leaf_prims(), osc.num_prims)
    for s, seed in ((0, 0), (5, 0x9E3779B9_00000005)):
        p = sc.params(64, s, 0, 50, seed)
        pix = pixel_seeds((p.height, p.width)).reshape(-1)
        rgb, rays, flags = osc.replay_paths(cam, p, pix, np.full(pix.size, s, np.int32), leaf)
        rgb, rays, flags = rgb.reshape(p.height, p.width, 3), rays.reshape(p.height, p.width), flags.reshape(p.height, p.width)
        assert (rgb > 0).any(axis=2).mean() > 0.5, "most paths must reach a light"
        for flag in (api.FLAG_BVH_LOCKSTEP, api.FLAG_BVH_PERSISTENT, api.FLAG_BVH_LOCKSTEP | api.FLAG_NO_TAIL):
            p = sc.params(64, s, flag, 50, seed)
            img, _, st = gsc.render(cam, p)
            ok, unfl = match(img, rgb, rays), flags == 0
            bad_unfl, bad_all = (~ok & unfl).sum() / max(1, unfl.sum()), (~ok).mean()
            label = f"depth-limit scene, flags {flag}, s={s}"
            print(f"[lbvh] {label}: mismatch unflagged {bad_unfl:.2e} all {bad_all:.2e}; flagged {(~unfl).mean():.4f}; "
                  f"rays {st.rays} replay {int(rays.sum())}")
            assert bad_unfl <= MAX_UNFLAGGED and bad_all <= MAX_ALL, label
            slack = np.maximum(rays, 50)[(~ok) | (~unfl)].sum()
            assert abs(int(st.rays) - int(rays.sum())) <= slack, label
    # feature buffers against the camera-ray and closest-hit hooks (test_gpu_aov.py)
    desc = sc.desc
    prims = gsc.prims()
    p = sc.params(64, 3)
    w, h = p.width, p.height
    albedo, normal, dist, hits, st = gsc.render_aov(cam, p)
    rows = np.arange(h - 1, -1, -1, dtype=np.uint32)[:, None]
    seeds = (rows * np.uint32(w) + np.arange(w, dtype=np.uint32)[None, :]).reshape(-1)
    cr = gsc.eval_camera_rays(cam, p, seeds, np.full(w * h, 3, np.int32))
    prim, tt, n3, ff, _ = gsc.trace_closest(cr, seed=0)
    hit = prim >= 0
    assert hit.all() and (hits.reshape(-1) == hit).all(), "every camera ray of the depth-limit scene hits a sphere"
    dn = np.abs(normal.reshape(-1, 3) - n3).max()
    assert dn <= 2.0 ** -21, f"normals differ from rt1w_trace_closest by {dn:.3e}"
    dd = cr["direction"].astype(np.float64)
    want = tt.astype(np.float64) * np.sqrt((dd * dd).sum(1))
    assert np.all(np.abs(dist.reshape(-1) - want) <= 1e-6 * want)
    mats = [desc.materials[i] for i in range(desc.n_materials)]
    tex_of = np.array([mats[prims[k].material].texture for k in prim], np.int32)
    colour = np.zeros((len(prim), 3), np.float32)
    for tx in np.unique(tex_of):  # solid colours: the device's texture value, wherever it is asked
        colour[tex_of == tx] = gsc.eval_texture(int(tx), np.zeros(((tex_of == tx).sum(), 3)))
    is_light = np.array([mats[prims[k].material].type == api.MAT_DIFFUSE_LIGHT for k in prim])
    want_alb = np.where(is_light[:, None], np.where(ff[:, None] != 0, np.clip(colour, 0, 1), 0), colour).astype(np.float32)
    assert np.array_equal(albedo.reshape(-1, 3), want_alb), "albedo differs from the material table"
    gsc.close()
