"""First-hit feature buffers (include/rt1w.h: rt1w_render_aov): albedo, normal, distance and hit count of the first segment
of every path, summed over the sample range.

- At one sample, every pixel against the camera-ray hook traced by rt1w_trace_closest: hits exact, normals bit-equal
  (on BVH scenes all but a few within 2 ulp: the f64 solve's FMA contraction is the compiler's), distances within 1e-6 relative, albedos as the material table says (texture lookups exact off cell borders).
- The same first segment as the render, media draws included: with max_depth = 1 a render sum equals the background
  exactly where the call counts no hit.
- Every kernel family (flat scan with and without media, binary and 8-wide tree), sample-range splits, determinism, a
  two-device context, the argument checks, the memory the call allocates (no path pool) and the demo driver's PFM files.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BACKGROUND = (0.25, 0.5, 0.125)


@pytest.fixture(scope="module")
def ctx(rt):
    c = rt.api.Context(0)
    yield c
    c.close()


def _n_gpus():
    import torch

    return torch.cuda.device_count()


def _params(api, hs, width, begin, end, seed=3, flags=0, max_depth=None, background=None):
    p = hs.params(width=width, sample_begin=begin, sample_end=end, seed=seed, flags=flags, max_depth=max_depth)
    if background is not None:
        p.background[:] = list(background)
    return p


def _seeds_top_down(w, h):
    """Pixel seeds j*w+i (row j counted from the bottom) in the outputs' order (row 0 = top)."""
    rows = np.arange(h - 1, -1, -1, dtype=np.uint32)[:, None]
    return (rows * np.uint32(w) + np.arange(w, dtype=np.uint32)[None, :]).reshape(-1)


HOOK_SCENES = [("cornel_box", {}, 96), ("two_spheres", {}, 96), ("earth", {}, 96), ("simple_light", {}, 96),
               ("stress", dict(stress_spheres=200_000), 160)]


@pytest.mark.parametrize("name,kw,width", HOOK_SCENES, ids=[s[0] for s in HOOK_SCENES])
def test_one_sample_matches_the_parity_hooks(rt, ctx, name, kw, width):
    api = rt.api
    hs = api.HostScene(name, seed=1, **kw)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    assert cam.lens_radius == 0.0, "the hook's f32 origin is exact for pinhole cameras only"
    desc = hs.desc.contents
    prims = gsc.prims()
    mats = [desc.materials[i] for i in range(desc.n_materials)]
    bg = np.clip(np.array(hs.settings.background[:], np.float32), 0, 1)
    for s in range(4):
        p = _params(api, hs, width, s, s + 1)
        w, h = p.width, p.height
        albedo, normal, dist, hits, st = gsc.render_aov(cam, p)
        assert st.paths == st.rays == w * h and st.waves == 0 and st.launches == 1
        rays = gsc.eval_camera_rays(cam, p, _seeds_top_down(w, h), np.full(w * h, s, np.int32))
        prim, t, n3, ff, uv = gsc.trace_closest(rays, seed=0)
        hit = prim >= 0
        label = f"{name} sample {s}"
        assert (hits.reshape(-1) == hit).all(), f"{label}: {np.sum(hits.reshape(-1) != hit)} pixels differ in hit / miss"
        assert 0.05 < hit.mean(), label
        # Normals: bit-equal on the flat scan.  On BVH scenes the f64 sphere solve is compiled into each kernel and left to the
        # compiler's FMA contraction (DESIGN.md sections 13-14), so the hook's kernel and this one may round a hit's t
        # differently in its last bits: the same primitive, a normal component 1-2 ulp apart.
        same_n = (normal.reshape(-1, 3) == n3).all(1)
        if gsc.info().n_wide_nodes == 0:
            assert same_n[hit].all(), f"{label}: normals differ from rt1w_trace_closest"
        else:
            dn = np.abs(normal.reshape(-1, 3)[hit] - n3[hit]).max(initial=0.0)
            print(f"{label}: {np.sum(hit & ~same_n)} of {hit.sum()} normals differ in their last bits, by at most {dn:.3e}")
            assert np.sum(hit & ~same_n) <= 5e-3 * hit.sum() and dn <= 2.0 ** -21, f"{label}: normals differ from rt1w_trace_closest"
        assert (normal.reshape(-1, 3)[~hit] == 0).all() and (dist.reshape(-1)[~hit] == 0).all()
        d = rays["direction"].astype(np.float64)
        want = t.astype(np.float64) * np.sqrt((d * d).sum(1))
        got = dist.reshape(-1).astype(np.float64)
        assert np.all(np.abs(got[hit] - want[hit]) <= 1e-6 * want[hit]), f"{label}: distance off by {np.max(np.abs(got[hit] / want[hit] - 1)):.2e}"
        # albedo by material
        alb = albedo.reshape(-1, 3)
        assert (alb[~hit] == bg).all(), f"{label}: a miss must see the clamped background"
        mat_of = np.array([mats[prims[k].material].type if k >= 0 else -1 for k in prim], np.int32)
        tex_of = np.array([mats[prims[k].material].texture if k >= 0 else -1 for k in prim], np.int32)
        o = rays["origin"].astype(np.float64)
        pts = o + t.astype(np.float64)[:, None] * d
        want_alb = np.zeros_like(alb)
        for tex in np.unique(tex_of[hit & np.isin(mat_of, [api.MAT_LAMBERTIAN, api.MAT_DIFFUSE_LIGHT])]):
            sel = hit & (tex_of == tex) & np.isin(mat_of, [api.MAT_LAMBERTIAN, api.MAT_DIFFUSE_LIGHT])
            want_alb[sel] = gsc.eval_texture(int(tex), pts[sel], uv[sel])
        light = hit & (mat_of == api.MAT_DIFFUSE_LIGHT)
        want_alb[light] = np.where(ff[light, None] != 0, np.clip(want_alb[light], 0, 1), 0)
        metal = hit & (mat_of == api.MAT_METAL)
        want_alb[metal] = np.array([mats[prims[k].material].albedo[:] for k in prim[metal]], np.float32).reshape(-1, 3)
        want_alb[hit & (mat_of == api.MAT_DIELECTRIC)] = 1.0
        want_alb[~hit] = bg
        lam = hit & (mat_of == api.MAT_LAMBERTIAN)
        solid = np.array([desc.textures[k].type == api.TEX_SOLID if k >= 0 else True for k in tex_of])
        exact = ~lam | solid
        assert np.array_equal(alb[exact], want_alb[exact]), f"{label}: albedo differs from the material table"
        # checker, image and noise textures: the hook's hit point carries the f32 rounding of t, so checker cells may flip at
        # their borders and noise values move in their last bits
        off = ~np.isclose(alb[~exact], want_alb[~exact], rtol=0.0, atol=1e-4).all(1)
        assert off.sum() <= 2e-3 * off.size, f"{label}: {off.sum()} of {off.size} textured albedos differ"
    gsc.close()


def _fog_scene(api):
    """Two ConstantMedium volumes (a sphere and a box) against the sky: a miss means the free-flight draw let the ray through."""
    b = api.DescBuilder()
    a, c, none = b.solid(0.8, 0.3, 0.2), b.solid(0.2, 0.4, 0.9), b.null_material()  # (a boundary's own material is never read)
    m1 = b.constant_medium(b.sphere((0.0, 0.0, -1.0), 0.6, none), 1.2, a)
    m2 = b.constant_medium(b.aabox((0.4, -0.5, -2.0), (1.4, 0.5, -1.0), none), 0.7, c)
    b.set_world(b.bvh([m1, m2]))
    cam = api.camera_new([0.0, 0.2, 1.5], [0.2, 0.0, -1.2], [0.0, 1.0, 0.0], 45.0, 1.5, 0.0, 2.5, 0.0, 1.0)
    return b, cam


SEGMENT_SCENES = ["fog", "cornel_smoke", "final_scene", "one_weekend"]


@pytest.mark.parametrize("name", SEGMENT_SCENES)
def test_same_first_segment_as_the_render(rt, ctx, name):
    """max_depth = 1: a path ends after its first closest hit, so its render sum is the background exactly when it missed."""
    api = rt.api
    if name == "fog":
        b, cam = _fog_scene(api)
        gsc = api.Scene(ctx, b.desc())
        make = lambda s: _fog_params(api, s)
    else:
        hs = api.HostScene(name, seed=1)
        gsc = api.Scene(ctx, hs.desc)
        cam = hs.camera()
        make = lambda s: _params(api, hs, 120, s, s + 1, max_depth=1, background=BACKGROUND)
    bg = np.array(BACKGROUND, np.float32)
    for s in range(8):
        p = make(s)
        rgb, _, _ = gsc.render(cam, p)
        _, _, _, hits, _ = gsc.render_aov(cam, p)
        sky = (rgb == bg).all(-1)
        bad = sky != (hits == 0)
        if name == "fog":
            assert 0.01 < (hits > 0).mean() and 0.01 < sky.mean(), "the fog scene must show hits and misses"
        assert not bad.any(), f"{name} sample {s}: {bad.sum()} pixels where render and feature buffers disagree on the first hit"
    gsc.close()


def _fog_params(api, s):
    p = api.RenderParams()
    p.width, p.height, p.sample_begin, p.sample_end, p.max_depth, p.seed = 120, 80, s, s + 1, 1, 11
    p.background[:] = list(BACKGROUND)
    return p


def _oracle_means(api, gsc, osc, hs, cam, w, h, spp, rng_seed):
    """Per-pixel means of the feature buffers from the oracle's closest hits: camera rays of camera.rs:61-73 drawn with numpy
    (jitter, lens disk, shutter time) - an independent sampler of the same distribution - traced by the oracle; albedos
    from the material table and the device texture hook (held against the oracle pointwise in test_gpu_shading_hooks)."""
    rng = np.random.default_rng(rng_seed)
    jj, ii = np.meshgrid(np.arange(h - 1, -1, -1), np.arange(w), indexing="ij")  # row 0 = top
    ii, jj = np.repeat(ii.reshape(-1), spp), np.repeat(jj.reshape(-1), spp)
    n = ii.size
    u, v = (ii + rng.random(n)) / (w - 1), (jj + rng.random(n)) / (h - 1)
    r, a = np.sqrt(rng.random(n)), 2.0 * np.pi * rng.random(n)
    lx, ly = cam.lens_radius * r * np.cos(a), cam.lens_radius * r * np.sin(a)
    c = {k: np.array(getattr(cam, k)[:]) for k in ("origin", "lower_left_corner", "horizontal", "vertical", "u", "v")}
    off = lx[:, None] * c["u"] + ly[:, None] * c["v"]
    rays = np.empty(n, dtype=api.RAY_DTYPE)
    rays["origin"] = c["origin"] + off
    rays["direction"] = c["lower_left_corner"] + u[:, None] * c["horizontal"] + v[:, None] * c["vertical"] - c["origin"] - off
    rays["time"] = cam.time0 + (cam.time1 - cam.time0) * rng.random(n)
    prim, t, normal, ff, uv, _ = osc.trace_closest(rays, seed=rng_seed)
    prims, desc = gsc.prims(), hs.desc.contents
    hit = prim >= 0
    kind = np.array([prims[k].kind if k >= 0 else -1 for k in prim])
    mat = np.array([prims[k].material if k >= 0 else -1 for k in prim])
    mtype = np.array([desc.materials[m].type if m >= 0 else -1 for m in mat])
    alb = np.zeros((n, 3))
    alb[~hit] = np.clip(np.array(hs.settings.background[:]), 0, 1)
    d = rays["direction"].astype(np.float64)
    pts = rays["origin"].astype(np.float64) + t[:, None] * d
    for m in np.unique(mat[hit]):
        sel = hit & (mat == m)
        mm = desc.materials[m]
        if mm.type in (api.MAT_LAMBERTIAN, api.MAT_ISOTROPIC, api.MAT_DIFFUSE_LIGHT):
            val = gsc.eval_texture(mm.texture, pts[sel], uv[sel].astype(np.float32)).astype(np.float64)
            if mm.type == api.MAT_DIFFUSE_LIGHT:
                val = np.where(ff[sel, None] != 0, np.clip(val, 0, 1), 0)
            alb[sel] = val
        elif mm.type == api.MAT_METAL:
            alb[sel] = np.array(mm.albedo[:])
        elif mm.type == api.MAT_DIELECTRIC:
            alb[sel] = 1.0
    medium = kind == api.NODE_CONSTANT_MEDIUM
    nrm = np.where((hit & ~medium)[:, None], normal, 0.0)
    dist = np.where(hit, t * np.sqrt((d * d).sum(1)), 0.0)
    per = lambda x: x.reshape(h, w, spp, -1).sum(2)
    hits = per(hit.astype(np.float64))[..., 0]
    return api.aov_means(per(alb), per(nrm), per(dist)[..., 0], hits, spp)


@pytest.mark.parametrize("name", ["cornel_box", "cornel_smoke", "final_scene", "one_weekend"])
def test_means_against_the_oracle(rt, ctx, oracle, name):
    """RMSE(gpu, oracle) <= 1.15 x RMSE(oracle, oracle') + 1e-3 for the mean albedo, normal and distance (section 3's bar)."""
    api = rt.api
    hs = api.HostScene(name, seed=1)
    gsc, osc = api.Scene(ctx, hs.desc), oracle.OracleScene(hs.desc)
    cam = hs.camera()
    w, spp = 128, 32
    p = _params(api, hs, w, 0, spp)
    h = p.height
    gpu = api.aov_means(*gsc.render_aov(cam, p)[:4], spp)
    o1, o2 = _oracle_means(api, gsc, osc, hs, cam, w, h, spp, 1), _oracle_means(api, gsc, osc, hs, cam, w, h, spp, 2)
    rmse = lambda a, b: float(np.sqrt(np.mean((np.asarray(a, np.float64) - b) ** 2)))
    for label, g, a, b in zip(("albedo", "normal", "distance"), gpu, o1, o2):
        e, base = rmse(g, a), rmse(a, b)
        print(f"{name} {label}: RMSE(gpu, oracle) {e:.4g}, RMSE(oracle, oracle') {base:.4g}")
        assert e <= 1.15 * base + 1e-3, f"{name} {label}: RMSE {e:.4g} against the oracle's own {base:.4g}"
    gsc.close()


def test_binary_and_wide_trees_agree(rt, ctx):
    api = rt.api
    hs = api.HostScene("stress", seed=1, stress_spheres=200_000)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    out = [gsc.render_aov(cam, _params(api, hs, 256, 0, 4, flags=f))[:4] for f in (api.FLAG_BVH_BINARY, api.FLAG_BVH_WIDE)]
    same = np.ones(out[0][3].shape, bool)
    for a, b in zip(out[0], out[1]):
        same &= (a == b).reshape(same.shape + (-1,)).all(-1)
    print(f"binary vs wide: {np.sum(~same)} of {same.size} pixels differ (distance ties)")
    assert same.mean() >= 0.999
    gsc.close()


def _close(a, b, n, label, hits=None):
    """Sums of n samples added in another order: within n*2^-22 of the sum of the contributions' magnitudes.  Albedo and
    distance contributions are >= 0, so that is the larger sum; a normal's components have |x| <= 1 and cancel, so their
    bound is the hit count (pass `hits`)."""
    mag = np.maximum(np.abs(a), np.abs(b))
    if hits is not None:
        mag = np.maximum(mag, np.asarray(hits, np.float64)[..., None])
    tol = n * 2.0 ** -22 * mag
    assert np.all(np.abs(a.astype(np.float64) - b) <= tol), f"{label}: off by {np.max(np.abs(a.astype(np.float64) - b) - tol):.3e} beyond n*2^-22"


@pytest.mark.parametrize("name,width", [("cornel_smoke", 64), ("final_scene", 64), ("cornel_box", 48)])
def test_sample_ranges_add_and_calls_repeat(rt, ctx, name, width):
    api = rt.api
    hs = api.HostScene(name, seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    whole = gsc.render_aov(cam, _params(api, hs, width, 0, 8))
    again = gsc.render_aov(cam, _params(api, hs, width, 0, 8))
    for a, b in zip(whole[:4], again[:4]):
        assert a.tobytes() == b.tobytes(), f"{name}: two calls differ"
    parts = [gsc.render_aov(cam, _params(api, hs, width, b, e)) for b, e in ((0, 4), (4, 8))]
    assert np.array_equal(parts[0][3] + parts[1][3], whole[3]), f"{name}: hit counts"
    for k, label in enumerate(("albedo", "normal", "distance")):
        _close(parts[0][k] + parts[1][k], whole[k], 8, f"{name} {label}", hits=whole[3] if label == "normal" else None)
    # many samples on a small image: several lanes share a pixel
    p = _params(api, hs, 32, 0, 512)
    a, b = gsc.render_aov(cam, p), gsc.render_aov(cam, p)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a[:4], b[:4]))
    assert (a[3] <= 512).all() and a[4].paths == 32 * p.height * 512
    gsc.close()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_devices_give_the_same_buffers(rt, ctx):
    api = rt.api
    hs = api.HostScene("cornel_smoke", seed=1)
    cam = hs.camera()
    one = api.Scene(ctx, hs.desc)
    c2 = api.Context([0, 1])
    two = api.Scene(c2, hs.desc)
    for begin, end in ((5, 6), (0, 9)):
        p = _params(api, hs, 64, begin, end)
        a, b = one.render_aov(cam, p), two.render_aov(cam, p)
        assert b[4].paths == a[4].paths
        assert np.array_equal(a[3], b[3])
        for k in range(3):
            if end - begin == 1:
                assert np.array_equal(a[k], b[k]), "1 spp: bit for bit"
            else:
                _close(a[k], b[k], end - begin, f"two devices, buffer {k}", hits=a[3] if k == 1 else None)
    two.close(), c2.close(), one.close()


def test_argument_checks(rt, ctx):
    api = rt.api
    lib = api.load_library()
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    for p in (_params(api, hs, 16, 0, 1, flags=api.FLAG_STATS), _params(api, hs, 16, 3, 3), _params(api, hs, 16, 0, 1)):
        if p.sample_end == 1 and not p.flags:
            p.width = 0
        with pytest.raises(api.Rt1wError) as e:
            gsc.render_aov(cam, p)
        assert e.value.status == api.ERR_INVALID
    p = _params(api, hs, 16, 0, 1)
    assert lib.rt1w_render_aov(gsc._h, C.byref(cam), C.byref(p), None, None, None, None, None) == api.ERR_INVALID
    hits = np.empty((p.height, p.width), np.float32)
    assert lib.rt1w_render_aov(gsc._h, C.byref(cam), C.byref(p), None, None, None, hits.ctypes.data, None) == api.OK
    assert hits.max() == 1.0
    with pytest.raises(api.Rt1wError):
        gsc.eval_camera_rays(cam, p, np.array([p.width * p.height], np.uint32), np.array([0], np.int32))
    gsc.close()


def test_allocates_no_path_pool(rt):
    """A first call on a fresh context at 3840x2160 takes its 8*W*H floats and little else (a render would allocate its queues)."""
    import torch

    api = rt.api
    c = api.Context(0)
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(c, hs.desc)
    p = _params(api, hs, 3840, 0, 1)
    p.height = 2160
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    _, _, _, hits, st = gsc.render_aov(hs.camera(), p)
    free1 = torch.cuda.mem_get_info(0)[0]
    grew = free0 - free1
    buffers = 8 * 4 * 3840 * 2160
    print(f"free device memory fell by {grew / 2**20:.1f} MiB for {buffers / 2**20:.1f} MiB of buffers")
    assert grew <= buffers + (64 << 20)
    assert st.paths == 3840 * 2160 and hits.max() == 1.0
    gsc.close()
    c.close()


def test_demo_driver_writes_pfm_files(rt, ctx):
    api = rt.api
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "rt1w_main")
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "P")
        r = subprocess.run([exe, "cornel_box", "--width", "64", "--spp", "4", "--aov", prefix], capture_output=True, timeout=300)
        assert r.returncode == 0, r.stderr.decode()
        assert r.stdout.startswith(b"P3")
        files = {k: api.read_pfm(f"{prefix}.{k}.pfm") for k in ("color", "albedo", "normal", "distance")}
        bad = subprocess.run([exe, "cornel_box", "--width", "8", "--spp", "2", "--frames", "2", "--aov", prefix], capture_output=True, timeout=60)
        assert bad.returncode == 2
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    p = hs.params(width=64, spp=4, seed=0)
    albedo, normal, dist, hits, _ = gsc.render_aov(hs.camera(), p)
    want = api.aov_means(albedo, normal, dist, hits, 4)
    for k, arr in zip(("albedo", "normal", "distance"), want):
        assert files[k].shape == arr.shape and files[k].tobytes() == arr.tobytes(), f"{k}.pfm differs from the binding's means"
    rgb, _, _ = gsc.render(hs.camera(), p)
    assert files["color"].shape == rgb.shape and np.isfinite(files["color"]).all()
    assert np.allclose(files["color"], np.nan_to_num(rgb, nan=0.0) / 4, rtol=1e-5, atol=1e-6)
    gsc.close()


def test_pfm_round_trip(rt, tmp_path):
    api = rt.api
    rng = np.random.default_rng(1)
    for shape in ((5, 7, 3), (4, 6)):
        a = rng.standard_normal(shape).astype(np.float32)
        path = str(tmp_path / "x.pfm")
        api.write_pfm(path, a)
        assert open(path, "rb").read(2) == (b"PF" if len(shape) == 3 else b"Pf")
        assert np.array_equal(api.read_pfm(path), a)
