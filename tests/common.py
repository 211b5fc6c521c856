"""Shared helpers of the parity tests: the fixed synthetic ray set (SURVEY.md §8d) and image statistics."""
import numpy as np

RAY_SEED = 0xC0FFEE


def scene_bounds(prims):
    lo = np.min([list(p.bbox_min) for p in prims], axis=0)
    hi = np.max([list(p.bbox_max) for p in prims], axis=0)
    return lo, hi


def uniform_sphere(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def cosine_about(rng, normals):
    """Cosine-distributed directions about unit normals (math.rs:39-49 in an arbitrary frame)."""
    n = normals.shape[0]
    r1, r2 = rng.random(n), rng.random(n)
    phi = 2 * np.pi * r1
    local = np.stack([np.cos(phi) * np.sqrt(r2), np.sin(phi) * np.sqrt(r2), np.sqrt(1 - r2)], axis=1)
    a = np.where(np.abs(normals[:, :1]) > 0.9, np.array([[0.0, 1.0, 0.0]]), np.array([[1.0, 0.0, 0.0]]))
    v = np.cross(normals, a)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    u = np.cross(normals, v)
    return local[:, :1] * u + local[:, 1:2] * v + local[:, 2:3] * normals


def make_ray_set(api, host_scene, oracle_scene, prims, n, max_extent=None, aspect=None):
    """Half uniform rays in the inflated scene box, a quarter camera rays, a quarter secondary rays."""
    rng = np.random.Generator(np.random.Philox(RAY_SEED))
    lo, hi = scene_bounds(prims)
    if max_extent is not None:  # scenes with a huge fog/ground sphere: sample around the camera target instead
        ctr = np.array(list(host_scene.settings.look_at))
        lo, hi = np.maximum(lo, ctr - max_extent), np.minimum(hi, ctr + max_extent)
    ext = hi - lo
    lo, hi = lo - 0.1 * ext, hi + 0.1 * ext
    n_uni, n_cam = n // 2, n // 4
    n_sec = n - n_uni - n_cam
    rays = np.zeros(n, dtype=api.RAY_DTYPE)
    # uniform
    rays["origin"][:n_uni] = lo + rng.random((n_uni, 3)) * (hi - lo)
    rays["direction"][:n_uni] = uniform_sphere(rng, n_uni) * (0.5 + 19.5 * rng.random((n_uni, 1)))
    # camera rays on a regular (s, t) grid (camera.rs:67-70 with lens radius 0)
    cam = host_scene.camera() if aspect is None else host_scene.camera(aspect=aspect)  # aspect: what Camera::new is given (camera.rs:27)
    side = int(np.ceil(np.sqrt(n_cam)))
    s, t = np.meshgrid((np.arange(side) + 0.5) / side, (np.arange(side) + 0.5) / side)
    s, t = s.ravel()[:n_cam], t.ravel()[:n_cam]
    origin = np.array(list(cam.origin))
    llc, hor, ver = np.array(list(cam.lower_left_corner)), np.array(list(cam.horizontal)), np.array(list(cam.vertical))
    rays["origin"][n_uni:n_uni + n_cam] = origin
    rays["direction"][n_uni:n_uni + n_cam] = llc + s[:, None] * hor + t[:, None] * ver - origin
    rays["time"] = rng.random(n).astype(np.float32)
    # secondary rays: from the oracle's hit points of (a resampling of) the camera rays
    idx = n_uni + rng.integers(0, n_cam, n_sec)
    prim, tt, normal, _, _, _ = oracle_scene.trace_closest(rays[idx], seed=1)
    ok = prim >= 0
    o = rays["origin"][idx].astype(np.float64) + np.where(ok, tt, 0.0)[:, None] * rays["direction"][idx].astype(np.float64)
    nrm = np.where(ok[:, None], normal, np.array([[0.0, 1.0, 0.0]]))
    nrm = nrm / np.linalg.norm(nrm, axis=1, keepdims=True)
    rays["origin"][n_uni + n_cam:] = o
    rays["direction"][n_uni + n_cam:] = cosine_about(rng, nrm)
    return rays


def quantise(rgb_sum, spp):
    """Display for SampledColor (color.rs:56-65) in numpy."""
    x = np.where(np.isnan(rgb_sum), 0.0, rgb_sum) / spp
    g = np.clip(np.sqrt(np.maximum(x, 0.0)), 0.0, 0.999)
    return (256.0 * g).astype(np.int64)


def check_trace_parity(gsc, osc, rays, seed=0x5EED, max_ambiguous=0.02, min_hit_fraction=0.1, label="", cache=None):
    """north_star checks 1 and 2 on one ray set: primitive ids bit-exact on every ray the oracle does not tag as a tie,
    hit distance <= 1e-5 relative, normal <= 1e-5, (u, v) <= 2e-5, front_face equal, misses report t = inf.
    Prints the ambiguous fraction (pytest -s / -rP shows it) and returns it.
    cache: a dict that keeps the oracle's answers between calls on the same rays (several device scenes, one oracle)."""
    n = len(rays)
    gp, gt, gn, gff, guv = gsc.trace_closest(rays, seed=seed)
    if cache is not None and "trace" in cache:
        op, ot, on, off, ouv, amb = cache["trace"]
    else:
        op, ot, on, off, ouv, amb = osc.trace_closest(rays, seed=seed)
        if cache is not None:
            cache["trace"] = (op, ot, on, off, ouv, amb)
    keep = amb == 0
    frac_amb = 1.0 - keep.mean()
    print(f"[trace parity] {label}: {n} rays, {frac_amb:.5f} ambiguous (ties within 1e-9 relative), {(op >= 0).mean():.3f} hit")
    assert frac_amb <= max_ambiguous, f"{frac_amb:.4f} of the rays are ambiguous: the ray set is badly conditioned"
    bad = keep & (gp != op)
    assert not bad.any(), f"{bad.sum()} primitive-id mismatches, first at ray {np.flatnonzero(bad)[:5]}: gpu {gp[bad][:5]} oracle {op[bad][:5]}"
    hit = keep & (op >= 0)
    assert hit.sum() >= min_hit_fraction * n
    rel_t = np.abs(gt[hit].astype(np.float64) - ot[hit]) / np.maximum(np.abs(ot[hit]), 1e-30)
    assert rel_t.max() <= 1e-5, f"hit distance off by {rel_t.max():.3e} relative"
    dn = np.abs(gn[hit].astype(np.float64) - on[hit]).max()
    assert dn <= 1e-5, f"normal off by {dn:.3e}"
    assert (gff[hit] == off[hit]).all()
    du = np.abs(guv[hit, 0].astype(np.float64) - ouv[hit, 0])
    du = np.minimum(du, 1.0 - du)  # u wraps at the atan2 branch cut (math.rs:69)
    dv = np.abs(guv[hit, 1].astype(np.float64) - ouv[hit, 1])
    assert max(du.max(), dv.max()) <= 2e-5
    miss = keep & (op < 0)
    assert np.isinf(gt[miss]).all()
    return frac_amb


def _stats(stat, n):
    mean = stat[..., :3] / n
    var = np.maximum(stat[..., 3:] / n - mean * mean, 0.0)
    return mean, var


def check_render_parity(api, gsc, osc, cam, make_params, spp, stat_clamp=20.0, flags=0, cache=None):
    """north_star check 3 (different RNG streams, so statistical): >= 99.9 % of the pixel-channel means within 5 sigma of
    the oracle's, RMSE(gpu, oracle) <= 1.15 RMSE(oracle, oracle') + 0.5 8-bit level, image mean and rays/path within 2 %.
    make_params(spp, sample_begin, flags, stat_clamp, seed) -> RenderParams."""
    p = make_params(spp, 0, api.FLAG_STATS | flags, stat_clamp, 3)
    g_sum, g_stat, g_st = gsc.render(cam, p, want_stat=True)
    assert g_st.paths == p.width * p.height * spp
    if cache is not None and "render" in cache:  # several device renders (kernels, builders) against one pair of oracle images
        oa_stat, oa_st, ob_stat = cache["render"]
    else:
        oa_sum, oa_stat, oa_st = osc.render(cam, p, want_stat=True)
        pb = make_params(2 * spp, spp, api.FLAG_STATS, stat_clamp, 0)
        ob_sum, ob_stat, _ = osc.render(cam, pb, want_stat=True)
        if cache is not None:
            cache["render"] = (oa_stat, oa_st, ob_stat)
    gm, gv = _stats(g_stat.astype(np.float64), spp)
    am, av = _stats(oa_stat, spp)
    bm, _ = _stats(ob_stat, spp)
    sigma = np.sqrt((gv + av) / spp) + 1e-4
    z = np.abs(gm - am) / sigma
    frac_ok = (z <= 5.0).mean()
    assert frac_ok >= 0.999, f"only {frac_ok:.5f} of the pixel means are within 5 sigma (worst z = {z.max():.1f})"
    img_g, img_a, img_b = (quantise(m, 1) for m in (gm, am, bm))
    rmse_ga = np.sqrt(np.mean((img_g - img_a) ** 2.0))
    rmse_ab = np.sqrt(np.mean((img_a - img_b) ** 2.0))
    assert rmse_ga <= 1.15 * rmse_ab + 0.5, f"RMSE gpu-oracle {rmse_ga:.2f} vs oracle-oracle {rmse_ab:.2f} (8-bit levels)"
    # whole-image mean within 2 % (+ 4 sigma of the two estimates: scenes lit by rarely-found lights, like the stress scene,
    # have image means that are themselves noisy at test sizes)
    sigma_mean = np.sqrt((gv + av).sum() / spp) / gv.size
    assert abs(gm.mean() - am.mean()) <= 0.02 * am.mean() + 4.0 * sigma_mean + 1e-4, \
        f"image mean gpu {gm.mean():.5f} oracle {am.mean():.5f} (sigma of the difference {sigma_mean:.5f})"
    rpp_g, rpp_o = g_st.rays / g_st.paths, oa_st.rays / oa_st.paths
    assert abs(rpp_g - rpp_o) <= 0.02 * rpp_o, f"rays/path gpu {rpp_g:.3f} oracle {rpp_o:.3f}"
    return g_st, oa_st


def pixel_seeds(shape):
    """The reference pixel seed j*w+i (main.rs:964) of every pixel of an (h, w, ...) image: rows are stored top first."""
    h, w = shape[0], shape[1]
    rows = np.arange(h)[:, None]
    return (h - 1 - rows) * w + np.arange(w)[None, :]


def check_identical_sums(a, b, spp, label, sample_begin=0):
    """The sums of two schedules of the same paths (rgb_sum or stat: (h, w, k) float32 arrays, or frame-major stacks of them).
    Every path adds to its pixel with ONE atomic and the sums start at zero, so only the order of the additions may differ:
      * NaN (and inf) in exactly the same places;
      * spp == 1: every finite value bit for bit (0 + c is exact in any order);
      * spp == n > 1: every value within 2 n 2^-24 of its magnitude (all contributions are >= 0, so either order is within
        (n - 1) 2^-24 |sum| of the exact sum).
    On failure: the first pixels as (pixel seed, sample index at spp == 1) and both values in hex."""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    assert a.shape == b.shape, f"{label}: shapes {a.shape} and {b.shape}"
    nan_a, nan_b = np.isnan(a), np.isnan(b)
    if spp == 1:
        bad = (nan_a != nan_b) | (~nan_a & ~nan_b & (a.view(np.uint32) != b.view(np.uint32)))
        bar = "bit for bit"
    else:
        fin = np.isfinite(a) & np.isfinite(b)
        with np.errstate(invalid="ignore"):  # inf - inf: those pixels are judged above
            err = np.abs(a.astype(np.float64) - b.astype(np.float64))
        lim = 2.0 * spp * 2.0 ** -24 * np.maximum(np.abs(a), np.abs(b)).astype(np.float64)
        bad = (nan_a != nan_b) | (np.isinf(a) != np.isinf(b)) | (np.isinf(a) & (a != b)) | (fin & ~(err <= lim))
        bar = f"within 2*{spp}*2^-24 relative"
    if not bad.any():
        return
    bad_px = bad.reshape(-1, *a.shape[-3:]).any(axis=-1)  # (frames, h, w)
    n_px = int(bad_px.sum())
    seeds = pixel_seeds(a.shape[-3:])
    lines = []
    for f, row, col in np.argwhere(bad_px)[:5]:
        va, vb = a.reshape(-1, *a.shape[-3:])[f, row, col], b.reshape(-1, *a.shape[-3:])[f, row, col]
        where = f"frame {f}, " if bad_px.shape[0] > 1 else ""
        path = f"pixel seed {seeds[row, col]}" + (f", sample {sample_begin}" if spp == 1 else f", samples [{sample_begin}, {sample_begin + spp})")
        lines.append(f"  {where}{path}: {' '.join(f'{x:08x}' for x in va.view(np.uint32))} vs {' '.join(f'{x:08x}' for x in vb.view(np.uint32))}"
                     f" ({va.tolist()} vs {vb.tolist()})")
    raise AssertionError(f"{label}: {n_px} pixels differ (bar: {bar}); first ones:\n" + "\n".join(lines))


def check_identical_render(a, b, label, spp, sample_begin=0):
    """Two schedules of the same paths by the same kernels (wave capacity, tail-kernel take-over, sample ranges, batches,
    devices): the same paths, exactly the same rays, and sums and statistics as check_identical_sums allows - bit for bit
    at one sample per pixel.  a, b: (rgb_sum, stat or None, RenderStats)."""
    (ia, sta, sa), (ib, stb, sb) = a, b
    assert sa.paths == sb.paths, f"{label}: {sa.paths} vs {sb.paths} paths"
    check_identical_sums(ia, ib, spp, label, sample_begin)  # (before the ray count: a mismatch here names the paths)
    if sta is not None or stb is not None:
        check_identical_sums(sta, stb, spp, label + " (statistics)", sample_begin)
    assert sa.rays == sb.rays, f"{label}: {sa.rays} vs {sb.rays} rays"


def check_same_render(a, b, label=""):
    """Two renders of the same paths by two kernels that truly differ - lockstep / persistent BVH kernel, binary / 8-wide
    tree, LBVH / SAH builder: they visit primitives in another order and break ties between equal hit distances another way,
    and the persistent kernel builds its sines with sinf (FAST_SIN = false), so a handful of rays per million may go another
    way.  Schedules of the same kernels are compared bit for bit instead (check_identical_render).
    a, b: (rgb_sum, stat, RenderStats)."""
    (ia, _, sa), (ib, _, sb) = a, b
    assert sa.paths == sb.paths, label
    assert abs(float(sa.rays) - float(sb.rays)) <= 1e-4 * float(sa.rays), f"{label}: {sa.rays} vs {sb.rays} rays"
    ok = np.isfinite(ia) & np.isfinite(ib)
    close = np.isclose(ia, ib, rtol=1e-3, atol=1e-3) | ~ok
    assert close.all(axis=2).mean() >= 0.999, f"{label}: {(~close.all(axis=2)).sum()} pixels differ"
    assert abs(np.nansum(ia) - np.nansum(ib)) <= 2e-3 * abs(np.nansum(ia)), label


# --------------------------------------------------------------------------- BVH trees (test_host_bvh.py, test_gpu_lbvh.py)
def decode_wide(node):
    """Child boxes of one wide node as kernels.cuh: wide_visit sees them: origin + q * 2^(e - 127)."""
    step = np.ldexp(1.0, node["exp"].astype(np.int64) - 127)  # per axis
    lo = node["origin"].astype(np.float64)[:, None] + node["qlo"].astype(np.float64) * step[:, None]
    hi = node["origin"].astype(np.float64)[:, None] + node["qhi"].astype(np.float64) * step[:, None]
    return lo, hi  # [axis][slot]


def check_binary(t, lo, hi, max_depth_allowed=62):
    """A binary tree of single-primitive leaves (rt1w_build_bvh_host / _device output t over f64 boxes lo, hi): every primitive
    in exactly one leaf, sibling pairs at even indices, the depth t reports, at most max_depth_allowed levels (the traversal stack),
    and every node's f32 box strictly containing the f64 boxes below it.  Returns the number of nodes reached."""
    nodes, order = t["nodes"], t["prim_order"]
    n = len(lo)
    assert sorted(order.tolist()) == list(range(n))
    seen = np.zeros(n, dtype=np.int64)
    sub_lo, sub_hi = {}, {}
    stack, post = [(0, 0)], []
    depth = 0
    while stack:
        i, d = stack.pop()
        post.append(i)
        depth = max(depth, d)
        nd = nodes[i]
        if nd["count"] == 0:
            left = int(nd["left_first"])
            assert left >= 2 and left % 2 == 0 and left + 1 < len(nodes)  # sibling pairs, 64-byte aligned
            stack += [(left, d + 1), (left + 1, d + 1)]
        else:
            assert nd["count"] == 1  # single-primitive leaves (api.cu: kMaxLeaf)
            seen[int(nd["left_first"])] += 1
    assert (seen == 1).all(), "every primitive sits in exactly one leaf"
    assert depth == t["depth"] and t["depth"] <= max_depth_allowed
    for i in reversed(post):  # children before parents
        nd = nodes[i]
        if nd["count"] == 0:
            left = int(nd["left_first"])
            sub_lo[i], sub_hi[i] = np.minimum(sub_lo[left], sub_lo[left + 1]), np.maximum(sub_hi[left], sub_hi[left + 1])
        else:
            p = order[int(nd["left_first"])]
            sub_lo[i], sub_hi[i] = lo[p], hi[p]
        assert (nd["min"].astype(np.float64) < sub_lo[i]).all() and (nd["max"].astype(np.float64) > sub_hi[i]).all(), \
            "a node's f32 box strictly contains the f64 boxes below it (bvh.h: conservative_box)"
    return len(post)


def check_wide(t, lo, hi, max_wide_depth=10):
    """Its 8-wide collapse: every leaf slot one binary leaf, nodes in BFS order with adjacent children and primitives, empty
    slots unhittable, every decoded child box containing what lies below it, the wide depth t reports, at most
    max_wide_depth (kernels.cuh: kWideMaxDepth; deeper collapses keep the binary walk).  Returns the mean slots per node."""
    nodes, wide, order, remap = t["nodes"], t["wide_nodes"], t["prim_order"], t["wide_leaf_remap"]
    n = len(lo)
    assert sorted(remap.tolist()) == list(range(n))
    leaf_node_of = {int(nd["left_first"]): k for k, nd in enumerate(nodes) if nd["count"] != 0 and (k != 1)}
    next_child, next_prim, slots = 1, 0, 0
    queue, depth_of = [0], {0: 0}
    kids = {}  # wide node -> [(slot, child node or None, leaf or None)]
    for w in queue:  # breadth first = the order the builder emits children in
        nd = wide[w]
        imask, lmask = int(nd["imask"]), int(nd["leaf_mask"])
        assert imask & lmask == 0 and lmask < 256
        ni, nl = bin(imask).count("1"), bin(lmask).count("1")
        assert ni + nl >= 1 and (ni + nl >= 2 or len(wide) == 1)
        slots += ni + nl
        if ni:
            assert int(nd["child_base"]) == next_child  # a node's interior children are adjacent, nodes in BFS order
        if nl:
            assert int(nd["prim_base"]) == next_prim    # its leaf primitives are adjacent, in slot order
        ci = pi = 0
        kids[w] = []
        for s in range(8):
            if (imask >> s) & 1:
                child = next_child + ci
                ci += 1
                depth_of[child] = depth_of[w] + 1
                queue.append(child)
                kids[w].append((s, child, None))
            elif (lmask >> s) & 1:
                kids[w].append((s, None, next_prim + pi))
                pi += 1
            else:
                assert (nd["qlo"][:, s] == 255).all() and (nd["qhi"][:, s] == 0).all()  # empty slots can never be hit
        next_child += ni
        next_prim += nl
    # conservativeness, bottom-up: a slot's decoded box contains the binary leaf's f32 box (leaf slots) / every primitive
    # box below the child (interior slots)
    true_lo, true_hi = {}, {}
    for w in reversed(queue):
        clo, chi = decode_wide(wide[w])
        los, his = [], []
        for s, child, leaf in kids[w]:
            if leaf is not None:
                b = nodes[leaf_node_of[int(remap[leaf])]]
                assert (clo[:, s] <= b["min"]).all() and (chi[:, s] >= b["max"]).all(), "quantised box does not contain the leaf's f32 box"
                p = order[int(remap[leaf])]
                l, h = lo[p], hi[p]
            else:
                l, h = true_lo[child], true_hi[child]
            assert (clo[:, s] < l).all() and (chi[:, s] > h).all(), "quantised box does not contain what lies below it"
            los.append(l), his.append(h)
        true_lo[w], true_hi[w] = np.min(los, axis=0), np.max(his, axis=0)
    assert next_child == len(wide) and next_prim == n
    assert max(depth_of.values()) == t["wide_depth"] and t["wide_depth"] <= max_wide_depth
    return slots / len(wide)


def _slab(lo, hi, o, inv):
    a, b = (lo - o) * inv, (hi - o) * inv
    tn, tf = np.minimum(a, b).max(), np.maximum(a, b).min()
    return max(tn, 0.0) <= tf


def walk_binary(nodes, o, inv):
    out, stack = set(), [0]
    while stack:
        nd = nodes[stack.pop()]
        if not _slab(nd["min"].astype(np.float64), nd["max"].astype(np.float64), o, inv):
            continue
        if nd["count"] == 0:
            stack += [int(nd["left_first"]), int(nd["left_first"]) + 1]
        else:
            out.add(int(nd["left_first"]))
    return out


def walk_wide(wide, o, inv):
    out, stack = set(), [0]
    while stack:
        nd = wide[stack.pop()]
        clo, chi = decode_wide(nd)
        ci = pi = 0
        for s in range(8):
            interior, leaf = (int(nd["imask"]) >> s) & 1, (int(nd["leaf_mask"]) >> s) & 1
            hit = (interior or leaf) and _slab(clo[:, s], chi[:, s], o, inv)
            if interior:
                if hit:
                    stack.append(int(nd["child_base"]) + ci)
                ci += 1
            elif leaf:
                if hit:
                    out.add(int(nd["prim_base"]) + pi)
                pi += 1
    return out


def check_walks(t, lo, hi, seed=11, n_rays=None):
    """Reference walks in numpy: for random rays through the boxes' bounds, the set of leaves a slab walk of either tree
    reaches contains every primitive box the ray really enters (f64), so no closest hit can be culled.  Returns the most
    wide leaf slots one ray reaches and the number of primitive boxes the rays enter."""
    rng = np.random.Generator(np.random.Philox(seed))
    centre, ext = 0.5 * (lo.min(0) + hi.max(0)), (hi.max(0) - lo.min(0))
    leaf_of_prim_b = np.empty(len(lo), dtype=np.int64)
    leaf_of_prim_b[t["prim_order"]] = np.arange(len(lo))
    wide_leaf_of_binary = np.empty(len(lo), dtype=np.int64)
    wide_leaf_of_binary[t["wide_leaf_remap"]] = np.arange(len(lo))
    reached, most = 0, 0
    n_rays = n_rays or (40 if len(lo) > 1000 else 100)
    for _ in range(n_rays):
        o = centre + rng.uniform(-0.7, 0.7, 3) * ext
        d = rng.normal(size=3)
        d[np.abs(d) < 1e-3] = 1e-3
        inv = 1.0 / d
        a, b = (lo - o) * inv, (hi - o) * inv
        tn, tf = np.minimum(a, b).max(1), np.maximum(a, b).min(1)
        truly = set(np.flatnonzero(np.maximum(tn, 0.0) <= tf).tolist())  # primitive boxes the ray enters (f64)
        got_b = walk_binary(t["nodes"], o, inv)
        got_w = walk_wide(t["wide_nodes"], o, inv)
        assert {int(leaf_of_prim_b[p]) for p in truly} <= got_b
        assert {int(wide_leaf_of_binary[leaf_of_prim_b[p]]) for p in truly} <= got_w
        reached += len(truly)
        most = max(most, len(got_w))
    return most, reached
