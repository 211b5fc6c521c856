"""Edge-aware denoising (include/rt1w.h: rt1w_denoise, rt1w_render_denoised): the a-trous filter guided by the feature buffers.

- The kernels against `reference`, a numpy f64 restatement of the header's definition, on seeded synthetic sums (NaN and
  infinite sums, zero normals, misses, floored albedos) at 1x1 .. 255x129, K = 0..5, default and extreme sigmas.
  Bound: |out - ref| <= TOL(sigma_n) (|ref| + a_p max|I|), from f32 sums and the approximate division, square root, exp2 and
  log2 of the device (relative 2^-21 .. 2^-22 each); log2's absolute error is multiplied by sigma_n in the normal weight's
  exponent, hence the sigma_n term.  The observed maximum is printed.
- Exact properties: K = 0 gives C within 4 ulp, NaN sums give 0, out_rgb8 is the host resolve of out_rgb, regions bounded
  by normal or hit / miss edges do not see each other (bit for bit), a constant field stays constant, calls repeat.
- The fused call equals rt1w_denoise of its own noisy sums and a separate rt1w_render_aov, bit for bit, on every kernel
  family and on two devices; its paths and rays are rt1w_render's.
- Quality at 16 spp against a 2048-spp render with another seed, in 8-bit levels.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import check_identical_sums

gpu = pytest.mark.gpu

LUM = np.array([0.2126, 0.7152, 0.0722])
B3 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
DEFAULTS = (5, 4.0, 128.0, 1.0)  # iterations, sigma_luminance, sigma_normal, sigma_depth


def _shift(a, dy, dx):
    """b[y, x] = a[y + dy, x + dx] where that pixel exists (else 0) and the mask of where it does."""
    h, w = a.shape[:2]
    b, valid = np.zeros_like(a), np.zeros((h, w), bool)
    y0, y1, x0, x1 = max(0, -dy), min(h, h - dy), max(0, -dx), min(w, w - dx)
    if y0 < y1 and x0 < x1:
        b[y0:y1, x0:x1] = a[y0 + dy:y1 + dy, x0 + dx:x1 + dx]
        valid[y0:y1, x0:x1] = True
    return b, valid


def reference(rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits, n, iterations, sigma_l, sigma_n, sigma_z):
    """The header's definition in f64: -> (out_rgb[h,w,3], a[h,w,3], I[h,w,3] before the first pass)."""
    f = lambda x: np.asarray(x, np.float64)
    rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits = map(f, (rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits))
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        color = np.where(np.isfinite(rgb_sum), rgb_sum / n, 0.0)
        a = np.maximum(albedo_sum / n, 1e-3)
        irr = color / a
        m = stat[..., :3] / n
        v = np.maximum(stat[..., 3:] / n - m * m, 0.0) / (n - 1)
        v = np.where(np.isfinite(v), v, 0.0)
        var = ((LUM / a) ** 2 * v).sum(-1)
        nn = np.sqrt((normal_sum ** 2).sum(-1))
        nrm = np.where(nn[..., None] > 0, normal_sum / np.where(nn > 0, nn, 1.0)[..., None], 0.0)
        z = np.where(hits > 0, distance_sum / np.where(hits > 0, hits, 1.0), 0.0)
    irr0 = irr.copy()
    zp = np.pad(z, 1, mode="edge")
    gx, gy = (zp[1:-1, 2:] - zp[1:-1, :-2]) / 2, (zp[2:, 1:-1] - zp[:-2, 1:-1]) / 2
    nz = (nrm != 0).any(-1)

    def normal_test(dy, dx):  # -> (w_n, w_n > 0, tap exists)
        nq, valid = _shift(nrm, dy, dx)
        nzq, _ = _shift(nz, dy, dx)
        dot = (nrm * nq).sum(-1)
        both, none = nz & nzq, ~nz & ~nzq
        wn = np.where(none, 1.0, np.where(both, np.maximum(dot, 0.0) ** sigma_n, 0.0))
        passes = none | (both & ((sigma_n == 0) | (dot > 0)))
        return wn, passes, valid

    for k in range(iterations):
        s = 1 << k
        vs, vw = np.zeros_like(var), np.zeros_like(var)
        for j in (-1, 0, 1):
            for i in (-1, 0, 1):
                vq, valid = _shift(var, j, i)
                ok = valid if i == j == 0 else valid & normal_test(j, i)[1]
                kw = (2 - abs(i)) * (2 - abs(j))
                vs += np.where(ok, kw * vq, 0.0)
                vw += np.where(ok, kw, 0.0)
        g3 = vs / vw
        lum = irr @ LUM
        si, sw, sv = np.zeros_like(irr), np.zeros_like(var), np.zeros_like(var)
        for j in range(-2, 3):
            for i in range(-2, 3):
                iq, valid = _shift(irr, s * j, s * i)
                vq, _ = _shift(var, s * j, s * i)
                if i == j == 0:
                    w = np.ones_like(var)
                else:
                    zq, _ = _shift(z, s * j, s * i)
                    wn, _, _ = normal_test(s * j, s * i)
                    wz = np.exp(-np.abs(z - zq) / (sigma_z * np.abs(gx * s * i + gy * s * j) + 1e-3 * z + 1e-6))
                    wl = np.exp(-np.abs(lum - iq @ LUM) / (sigma_l * np.sqrt(g3) + 1e-6))
                    w = wn * wz * wl
                hw = np.where(valid, B3[i + 2] * B3[j + 2] * w, 0.0)
                si += hw[..., None] * iq
                sw += hw
                sv += hw * hw * vq
        irr, var = si / sw[..., None], sv / (sw * sw)
    return a * irr, a, irr0


def synthetic(rng, h, w, n, nan_fraction=0.01):
    """Sums of n samples with the structure of a render: smooth normals and distances with noise, misses (zero normal, no
    hit), medium-like hits (zero normal, hits), random normals, floored albedos, NaN and infinite colour sums."""
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    albedo = rng.uniform(0.02, 1.0, (h, w, 3))
    albedo[rng.random((h, w)) < 0.03] = rng.uniform(0.0, 1e-3, 3)
    irr = rng.uniform(0.0, 2.0, (h, w, 1)) * rng.uniform(0.5, 1.0, (h, w, 3))
    color = np.maximum(albedo * irr * (1.0 + 0.3 * rng.standard_normal((h, w, 3))), 0.0)
    sigma = color * rng.uniform(0.0, 1.5, (h, w, 3))
    rgb_sum = color * n
    stat = np.concatenate([rgb_sum, n * (color ** 2 + sigma ** 2)], axis=-1)
    normal = np.stack([np.sin(xx / 7.0), np.cos(yy / 5.0), np.ones((h, w))], -1) + 0.1 * rng.standard_normal((h, w, 3))
    kind = rng.random((h, w))
    normal[kind < 0.2] = rng.standard_normal((int((kind < 0.2).sum()), 3))
    z = 1.0 + xx / max(w, 1) + 0.5 * yy / max(h, 1) + 0.01 * rng.standard_normal((h, w))
    hits = rng.integers(1, n + 1, (h, w)).astype(np.float64)
    miss, medium = kind > 0.92, (kind > 0.88) & (kind <= 0.92)
    normal[miss | medium] = 0.0
    hits[miss] = 0.0
    normal_sum = normal * rng.uniform(0.2, 1.0, (h, w, 1)) * n
    distance_sum = np.where(hits > 0, z * hits, 0.0)
    bad = rng.random((h, w, 3))
    rgb_sum[bad < nan_fraction] = np.nan
    rgb_sum[bad > 1.0 - nan_fraction / 4] = np.inf
    f32 = lambda x: np.ascontiguousarray(x, np.float32)
    return tuple(f32(x) for x in (rgb_sum, stat, albedo * n, normal_sum, distance_sum, hits))


def tolerance(sigma_n):
    return 1e-4 * (1.0 + sigma_n / 500.0)


@pytest.fixture(scope="module")
def ctx(rt):
    c = rt.api.Context(0)
    yield c
    c.close()


def _dp(api, iterations, sigma_l, sigma_n, sigma_z):
    return api.DenoiseParams(iterations=iterations, sigma_luminance=sigma_l, sigma_normal=sigma_n, sigma_depth=sigma_z)


SIGMAS = [(4.0, 128.0, 1.0), (1e-3, 0.0, 1e-3), (1e3, 1e3, 1e3), (0.5, 1.0, 50.0)]
SIZES = [(1, 1), (1, 37), (37, 1), (64, 48), (255, 129)]  # (width, height)


@gpu
@pytest.mark.parametrize("width,height", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_kernel_against_the_restatement(rt, ctx, width, height):
    api = rt.api
    rng = np.random.default_rng(width * 1000 + height)
    worst = 0.0
    for n in (2, 16):
        sums = synthetic(rng, height, width, n)
        for iterations in range(6):
            for sig in (SIGMAS if iterations in (1, 5) else SIGMAS[:1]):
                out, rgb8 = ctx.denoise(*sums, n, _dp(api, iterations, *sig))
                want, a, irr0 = reference(*sums, n, iterations, *sig)
                scale = np.abs(want) + a * np.abs(irr0).max()
                err = np.abs(out - want) / scale
                worst = max(worst, float(err.max()))
                label = f"{width}x{height} n={n} K={iterations} sigmas={sig}"
                assert np.isfinite(out).all(), label
                assert err.max() <= tolerance(sig[1]), f"{label}: {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"
                assert np.array_equal(rgb8, api.resolve_rgb8(out, 1)), f"{label}: rgb8 is not the resolve of rgb"
    print(f"{width}x{height}: worst |out - ref| / (|ref| + a max|I|) = {worst:.3e}")


@gpu
def test_zero_passes_return_the_mean_and_nan_sums_give_zero(rt, ctx):
    api = rt.api
    rng = np.random.default_rng(7)
    n = 8
    sums = synthetic(rng, 40, 56, n, nan_fraction=0.05)
    out, _ = ctx.denoise(*sums, n, _dp(api, 0, *DEFAULTS[1:]))
    rgb_sum = sums[0].astype(np.float64)
    finite = np.isfinite(rgb_sum)
    assert (out[~finite] == 0).all(), "a non-finite sum must give 0"
    c = rgb_sum[finite] / n
    err = np.abs(out[finite] - c)
    assert np.all(err <= 4 * 2.0 ** -23 * np.abs(c)), f"K = 0: {np.max(err / np.maximum(np.abs(c), 1e-30)):.3e} relative"
    full, _ = ctx.denoise(*sums, n)
    assert (np.isfinite(full)).all()


def _halves(rng, h, w, n, kind):
    """Left and right halves separated by an edge: orthogonal normals (both halves hit) or hit / miss."""
    rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits = (x.copy() for x in synthetic(rng, h, w, n, nan_fraction=0.0))
    left = np.zeros((h, w), bool)
    left[:, : w // 2] = True
    normal_sum[left] = (n, 0.0, 0.0) if kind == "normals" else (0.5 * n, 0.2 * n, 0.8 * n)
    if kind == "normals":
        normal_sum[~left] = (0.0, 0.7 * n, 0.0)
        hits[:] = n
    else:
        normal_sum[~left], hits[~left] = 0.0, 0.0
        hits[left] = n
    distance_sum = np.where(hits > 0, 1.0 + 0.5 * rng.random((h, w)), 0.0).astype(np.float32) * hits
    return [rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits], left


@gpu
@pytest.mark.parametrize("kind", ["normals", "hit_miss"])
def test_edges_isolate_regions(rt, ctx, kind):
    """Changing the colour, statistics and albedo on one side of the edge - and, at a hit / miss edge, the distances - leaves
    every output pixel on the other side bit-identical, after 5 passes with steps up to 16."""
    rng = np.random.default_rng(11)
    h, w, n = 48, 64, 16
    base, left = _halves(rng, h, w, n, kind)
    out0, rgb80 = ctx.denoise(*base, n)
    for side in (left, ~left):
        pert = [x.copy() for x in base]
        for k in (0, 1, 2):
            noise = rng.uniform(0.1, 3.0, pert[k][side].shape).astype(np.float32)
            pert[k][side] = pert[k][side] * noise
        if kind == "hit_miss":
            pert[4][side] = pert[4][side] * np.float32(1.7)
        out1, rgb81 = ctx.denoise(*pert, n)
        other = ~side
        assert out1[other].tobytes() == out0[other].tobytes(), f"{kind}: the filter leaks across the edge"
        assert np.array_equal(rgb81[other], rgb80[other])
        assert not np.array_equal(out1[side], out0[side])


@gpu
@pytest.mark.parametrize("varying_albedo", [False, True], ids=["constant_colour", "constant_irradiance"])
def test_constant_field_stays_constant(rt, ctx, varying_albedo):
    """A constant colour (constant albedo), or a constant irradiance under a varying albedo, is left unchanged up to rounding
    (relative 1e-5: 5 passes of 25-tap f32 sums and the demodulation's approximate division), whatever the guides and the
    variance are."""
    rng = np.random.default_rng(5)
    h, w, n = 70, 90, 16
    rgb_sum, stat, albedo_sum, normal_sum, distance_sum, hits = synthetic(rng, h, w, n, nan_fraction=0.0)
    albedo = albedo_sum / n if varying_albedo else np.full((h, w, 3), (0.6, 0.4, 0.2), np.float32)
    albedo = np.maximum(albedo, 0.01)
    color = albedo * np.array([0.9, 1.3, 0.7], np.float32)
    out, _ = ctx.denoise((color * n).astype(np.float32), stat, (albedo * n).astype(np.float32), normal_sum, distance_sum, hits, n)
    rel = np.abs(out - color) / color
    print(f"constant field: worst relative change {rel.max():.3e}")
    assert rel.max() <= 1e-5


@gpu
def test_calls_repeat_bit_for_bit(rt, ctx):
    rng = np.random.default_rng(3)
    sums = synthetic(rng, 129, 255, 4)
    a, b = ctx.denoise(*sums, 4), ctx.denoise(*sums, 4)
    assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1])


# flat scan, flat scan with media, binary tree, 8-wide tree (and the media + rich textures of final_scene on both trees)
WIRING = [("cornel_box", {}, 0), ("cornel_smoke", {}, 0), ("final_scene", {}, "binary"), ("final_scene", {}, "wide"),
          ("stress", dict(stress_spheres=200_000), "binary"), ("stress", dict(stress_spheres=200_000), "wide")]


@gpu
@pytest.mark.parametrize("name,kw,tree", WIRING, ids=[f"{s[0]}-{s[2] or 'flat'}" for s in WIRING])
def test_fused_call_equals_the_three_calls(rt, ctx, name, kw, tree):
    api = rt.api
    hs = api.HostScene(name, seed=1, **kw)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    flags = {0: 0, "binary": api.FLAG_BVH_BINARY, "wide": api.FLAG_BVH_WIDE}[tree]
    p = hs.params(width=96, spp=8, seed=5, flags=flags, stat_clamp=8.0)
    dp = _dp(api, 4, 3.0, 64.0, 2.0)
    out, rgb8, rgb_sum, stat, st = gsc.render_denoised(cam, p, dp)
    albedo, normal, dist, hits, _ = gsc.render_aov(cam, p)
    want, want8 = ctx.denoise(rgb_sum, stat, albedo, normal, dist, hits, 8, dp)
    assert out.tobytes() == want.tobytes() and np.array_equal(rgb8, want8), f"{name} {tree}: fused call differs from the three calls"
    ps = hs.params(width=96, spp=8, seed=5, flags=flags | api.FLAG_STATS, stat_clamp=8.0)
    ref_sum, ref_stat, ref_st = gsc.render(cam, ps, want_stat=True)
    assert (st.paths, st.rays) == (ref_st.paths, ref_st.rays)
    check_identical_sums(rgb_sum, ref_sum, 8, f"{name} {tree} rgb_sum")
    check_identical_sums(stat, ref_stat, 8, f"{name} {tree} stat")
    assert st.launches >= ref_st.launches + 1 + 2 + 4 + 1
    gsc.close()


def _n_gpus():
    import torch

    return torch.cuda.device_count()


@gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_devices(rt, ctx):
    api = rt.api
    hs = api.HostScene("cornel_smoke", seed=1)
    cam = hs.camera()
    one = api.Scene(ctx, hs.desc)
    c2 = api.Context([0, 1])
    two = api.Scene(c2, hs.desc)
    p = hs.params(width=80, spp=9, seed=2, stat_clamp=8.0)
    out, rgb8, rgb_sum, stat, st = two.render_denoised(cam, p)
    aov = two.render_aov(cam, p)[:4]
    want, want8 = c2.denoise(rgb_sum, stat, *aov, 9)
    assert out.tobytes() == want.tobytes() and np.array_equal(rgb8, want8)
    ps = hs.params(width=80, spp=9, seed=2, flags=api.FLAG_STATS, stat_clamp=8.0)
    ref_sum, ref_stat, ref_st = one.render(cam, ps, want_stat=True)
    check_identical_sums(rgb_sum, ref_sum, 9, "two devices rgb_sum")
    check_identical_sums(stat, ref_stat, 9, "two devices stat")
    assert st.paths == ref_st.paths and st.rays == ref_st.rays
    two.close(), c2.close(), one.close()


QUALITY = [("cornel_box", 200), ("cornel_smoke", 200), ("final_scene", 200), ("one_weekend", 240)]


def _rmse(a8, b8):
    return float(np.sqrt(np.mean((a8.astype(np.float64) - b8) ** 2)))


@gpu
@pytest.mark.parametrize("name,width", QUALITY, ids=[q[0] for q in QUALITY])
def test_quality_at_16_spp(rt, ctx, name, width):
    """RMSE in 8-bit levels against a 2048-spp render with another seed: the denoised image is never worse than the noisy
    one, and on the Cornell box at most half of it."""
    api = rt.api
    hs = api.HostScene(name, seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    ref8, _ = gsc.render_rgb8(cam, hs.params(width=width, spp=2048, seed=99))
    p = hs.params(width=width, spp=16, seed=1)
    _, den8, rgb_sum, _, _ = gsc.render_denoised(cam, p)
    noisy, denoised = _rmse(api.resolve_rgb8(rgb_sum, 16), ref8), _rmse(den8, ref8)
    print(f"{name} {width}x{p.height} 16 spp: RMSE noisy {noisy:.2f}, denoised {denoised:.2f} levels (ratio {denoised / noisy:.3f})")
    assert denoised <= noisy, f"{name}: the filter made the image worse"
    if name == "cornel_box":
        assert denoised <= 0.5 * noisy
    gsc.close()


@gpu
def test_argument_checks(rt, ctx):
    api = rt.api
    lib = api.load_library()
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    sums = synthetic(np.random.default_rng(1), 8, 8, 4)
    ptrs = [s.ctypes.data for s in sums]
    out, rgb8 = np.empty((8, 8, 3), np.float32), np.empty((8, 8, 3), np.uint8)
    bad_params = [_dp(api, -1, 4, 128, 1), _dp(api, 11, 4, 128, 1), _dp(api, 5, 0, 128, 1), _dp(api, 5, 4, -1, 1), _dp(api, 5, 4, 128, 0),
                  _dp(api, 5, float("nan"), 128, 1), _dp(api, 5, 4, float("nan"), 1), _dp(api, 5, 4, 128, float("inf"))]
    den = lambda c, w, h, n, ins, dp, o, o8: lib.rt1w_denoise(c, w, h, n, *ins, dp, o, o8)
    assert den(ctx._h, 8, 8, 4, ptrs, None, out.ctypes.data, None) == api.OK
    assert den(ctx._h, 8, 8, 4, ptrs, C.byref(_dp(api, 10, 1e-6, 0, 1e6)), None, rgb8.ctypes.data) == api.OK
    for dp in bad_params:
        assert den(ctx._h, 8, 8, 4, ptrs, C.byref(dp), out.ctypes.data, None) == api.ERR_INVALID
    assert den(None, 8, 8, 4, ptrs, None, out.ctypes.data, None) == api.ERR_INVALID
    for k in range(6):
        assert den(ctx._h, 8, 8, 4, ptrs[:k] + [None] + ptrs[k + 1:], None, out.ctypes.data, None) == api.ERR_INVALID
    assert den(ctx._h, 8, 8, 4, ptrs, None, None, None) == api.ERR_INVALID
    assert den(ctx._h, 8, 8, 1, ptrs, None, out.ctypes.data, None) == api.ERR_INVALID
    assert den(ctx._h, 0, 8, 4, ptrs, None, out.ctypes.data, None) == api.ERR_INVALID
    p = hs.params(width=8, height=8, spp=4, seed=1)
    fused = lambda sc, cm, pp, dp, o, o8: lib.rt1w_render_denoised(sc, cm, pp, dp, o, o8, None, None, None)
    assert fused(gsc._h, C.byref(cam), C.byref(p), None, None, rgb8.ctypes.data) == api.OK
    assert fused(None, C.byref(cam), C.byref(p), None, out.ctypes.data, None) == api.ERR_INVALID
    assert fused(gsc._h, None, C.byref(p), None, out.ctypes.data, None) == api.ERR_INVALID
    assert fused(gsc._h, C.byref(cam), None, None, out.ctypes.data, None) == api.ERR_INVALID
    assert fused(gsc._h, C.byref(cam), C.byref(p), None, None, None) == api.ERR_INVALID
    for dp in bad_params:
        assert fused(gsc._h, C.byref(cam), C.byref(p), C.byref(dp), out.ctypes.data, None) == api.ERR_INVALID
    for change in (dict(sample_begin=3, sample_end=4), dict(sample_begin=2, sample_end=2), dict(width=0), dict(sample_begin=-1)):
        q = hs.params(width=8, height=8, spp=4, seed=1)
        for k, v in change.items():
            setattr(q, k, v)
        assert fused(gsc._h, C.byref(cam), C.byref(q), None, out.ctypes.data, None) == api.ERR_INVALID, change
    gsc.close()


@gpu
def test_demo_driver(rt, ctx):
    api = rt.api
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "rt1w_main")
    r = subprocess.run([exe, "cornel_box", "--width", "64", "--spp", "8", "--denoise"], capture_output=True, timeout=300)
    assert r.returncode == 0, r.stderr.decode()
    lines = r.stdout.decode().split("\n")
    assert lines[0] == "P3" and lines[1] == "64 64" and lines[2] == "255"
    body = np.array([int(x) for x in " ".join(lines[3:]).split()], np.int64)
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    p = hs.params(width=64, spp=8, seed=0)
    _, rgb8, _, _, _ = gsc.render_denoised(hs.camera(), p)
    assert body.shape == (64 * 64 * 3,)
    # (the demo's render sums are added in a schedule-dependent order: the filter may move a level where they round apart)
    assert np.mean(np.abs(body - rgb8.reshape(-1)) <= 1) > 0.99
    gsc.close()
    with tempfile.TemporaryDirectory() as d:
        for extra in (["--frames", "2"], ["--max-error", "2"], ["--aov", os.path.join(d, "P")]):
            bad = subprocess.run([exe, "cornel_box", "--width", "8", "--spp", "2", "--denoise"] + extra, capture_output=True, timeout=60)
            assert bad.returncode == 2, extra


def test_params_struct_matches_the_header(rt):
    """The ctypes mirror against the C compiler's sizeof and offsets, and DenoiseParams() against the documented defaults."""
    api = rt.api
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "rt1w.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\n", sizeof(rt1w_denoise_params), offsetof(rt1w_denoise_params, sigma_luminance),
         offsetof(rt1w_denoise_params, sigma_normal), offsetof(rt1w_denoise_params, sigma_depth), offsetof(rt1w_denoise_params, reserved));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(root, "include"), "-o", os.path.join(d, "p"), os.path.join(d, "p.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(d, "p")]).split()]
    M = api.DenoiseParams
    assert got == [C.sizeof(M), M.sigma_luminance.offset, M.sigma_normal.offset, M.sigma_depth.offset, M.reserved.offset]
    d = M()
    assert (d.iterations, d.sigma_luminance, d.sigma_normal, d.sigma_depth, d.reserved) == (*DEFAULTS, 0)


def test_restatement_basics():
    """The numpy restatement itself (no GPU): K = 0 is the mean, one pass of a constant field is the identity, a 1x1 image
    passes through, and an edge stops the filter."""
    rng = np.random.default_rng(2)
    n = 4
    sums = synthetic(rng, 12, 10, n, nan_fraction=0.0)
    out0, a, irr0 = reference(*sums, n, 0, 4.0, 128.0, 1.0)
    assert np.allclose(out0, sums[0] / n, rtol=1e-12)
    const = [x.copy() for x in sums]
    const[0][:] = 0.5 * n
    const[2][:] = 0.5 * n
    out, _, _ = reference(*const, n, 3, 4.0, 128.0, 1.0)
    assert np.allclose(out, 0.5, rtol=1e-12)
    one = [x[:1, :1] for x in sums]
    assert np.allclose(reference(*one, n, 5, 4.0, 128.0, 1.0)[0], one[0] / n, rtol=1e-12)
    edge = [x.copy() for x in sums]
    edge[3][:, :5] = (n, 0, 0)
    edge[3][:, 5:] = (0, n, 0)
    edge[5][:] = n
    base, _, _ = reference(*edge, n, 3, 4.0, 128.0, 1.0)
    edge[0][:, 5:] *= 3.0
    moved, _, _ = reference(*edge, n, 3, 4.0, 128.0, 1.0)
    assert np.array_equal(base[:, :5], moved[:, :5])
