"""Adaptive sampling (include/rt1w.h: rt1w_render_adaptive).  Sample s of pixel p is the same path whichever round renders
it, so every pixel that ends with n samples must hold what a uniform render of [0, n) gives it - sums, NaNs and statistics -
up to the order of the fp32 additions.  Also: the schedule, the convergence rule recomputed in numpy, the list shapes of
the wave kernels' pixel-list generation, the per-pixel resolve, the demo driver's --max-error and the argument checks."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CLAMP = 10.0  # stat_clamp of the renders below


def _schedule(min_spp, max_spp):
    s = [min_spp]
    while s[-1] < max_spp:
        s.append(min(2 * s[-1], max_spp))
    return s


def _rule_error(rgb_sum, stat, n):
    """The rule of rt1w.h in numpy: per pixel, the largest channel half-width in 8-bit levels (0 on NaN-sum channels)."""
    n = np.asarray(n, dtype=np.float64)[..., None]
    s1, s2 = stat[..., :3].astype(np.float64), stat[..., 3:].astype(np.float64)
    m = s1 / n
    v = np.fmax(s2 / n - m * m, 0.0) * n / (n - 1)
    se = np.sqrt(v / n)
    hi, lo = np.fmin(np.fmax(m + se, 0.0), 1.0), np.fmin(np.fmax(m - se, 0.0), 1.0)
    e = 128.0 * (np.sqrt(hi) - np.sqrt(lo))
    return np.where(np.isnan(rgb_sum), 0.0, e).max(axis=-1)


def _same_sums(a, b, label):
    assert (np.isnan(a) == np.isnan(b)).all(), f"{label}: NaN in different places"
    ok = ~np.isnan(a)
    np.testing.assert_allclose(a[ok], b[ok], rtol=1e-4, atol=1e-4, err_msg=label)


def _adaptive_vs_uniform(api, gsc, hs, width, min_spp, max_spp, max_error, flags=0, height=None, pool_paths=0, seed=7):
    """Adaptive render, then for every count n in out_spp the uniform [0, n) render: the pixels with count n must match it.
    -> (rgb_sum, spp, rgb8, stat, stats, {n: uniform (rgb_sum, stat, stats)})."""
    cam = hs.camera()
    p = hs.params(width=width, height=height, spp=max_spp, seed=seed, flags=flags, stat_clamp=CLAMP, pool_paths=pool_paths)
    rgb, spp, rgb8, stat, st = gsc.render_adaptive(cam, p, min_spp, max_error, want_stat=True)
    assert spp.shape == (p.height, p.width) and set(np.unique(spp)) <= set(_schedule(min_spp, max_spp))
    assert st.paths == int(spp.sum())
    uniform = {}
    for n in np.unique(spp):
        u = gsc.render(cam, hs.params(width=width, height=height, spp=int(n), seed=seed, flags=flags | api.FLAG_STATS, stat_clamp=CLAMP,
                                      pool_paths=pool_paths), want_stat=True)
        uniform[int(n)] = u
        m = spp == n
        _same_sums(rgb[m], u[0][m], f"sums of the pixels with {n} samples")
        np.testing.assert_allclose(stat[m], u[1][m], rtol=1e-4, atol=1e-4, err_msg=f"statistics of the pixels with {n} samples")
        assert np.array_equal(rgb8[m], api.resolve_rgb8(rgb, int(n))[m]), f"device resolve of the pixels with {n} samples"
    return rgb, spp, rgb8, stat, st, uniform


CASES = [  # scene, constructor arguments, width, flags: flat scan, flat + media, lockstep BVH, media + rich textures, persistent wide tree
    ("cornel_box", {}, 64, 0),
    ("cornel_smoke", {}, 64, 0),
    ("random_scene", {}, 96, 0),
    ("final_scene", {}, 64, 0),
    ("stress", dict(stress_spheres=200_000), 96, 0),
    ("random_scene", {}, 96, "persistent_binary"),
]


@pytest.mark.parametrize("name,kw,width,flags", CASES, ids=[f"{c[0]}-{c[3] or 'default'}" for c in CASES])
def test_adaptive_pixels_equal_uniform_renders(rt, gpu_ctx, name, kw, width, flags):
    api = rt.api
    if flags == "persistent_binary":
        flags = api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_BINARY
    hs = api.HostScene(name, seed=1, **kw)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, _, _, st, _ = _adaptive_vs_uniform(api, gsc, hs, width, 4, 64, 2.0, flags=flags)
    counts = np.unique(spp)
    print(f"[adaptive {name}] counts {dict(zip(counts.tolist(), np.bincount(np.searchsorted(counts, spp.ravel())).tolist()))}, "
          f"{st.paths} paths, {st.rays} rays")
    assert len(counts) >= 2, "the case should exercise more than one round"
    gsc.close()


def test_threshold_zero_runs_every_pixel_to_the_cap(rt, gpu_ctx):
    """max_error 0: every pixel gets max_spp, and the same paths trace the same rays as the uniform render."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, _, _, st, uni = _adaptive_vs_uniform(api, gsc, hs, 64, 4, 32, 0.0)
    assert (spp == 32).all() and st.rays == uni[32][2].rays
    gsc.close()


def test_huge_threshold_stops_every_pixel_at_min_spp(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, _, _, st, uni = _adaptive_vs_uniform(api, gsc, hs, 64, 8, 64, 1e9)
    assert (spp == 8).all() and st.rays == uni[8][2].rays
    gsc.close()


def test_the_rule_holds(rt, gpu_ctx):
    """Recomputed in numpy: a pixel that stopped before the cap meets the rule at its count; a pixel with more than min_spp
    samples failed it at the count before (uniform render of that count, with statistics).  The fp32 sums arrive in another
    order than in the render, so a few pixels within 1e-3 relative of the threshold may go either way."""
    api = rt.api
    min_spp, max_spp, thr = 4, 128, 1.0
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    rgb, spp, _, stat, _ = gsc.render_adaptive(cam, hs.params(width=64, spp=max_spp, seed=3, stat_clamp=CLAMP), min_spp, thr, want_stat=True)
    near_allowed = max(1, int(1e-3 * spp.size))
    e = _rule_error(rgb, stat, spp)
    stopped = spp < max_spp
    bad = stopped & ~(e <= thr)
    assert bad.sum() <= near_allowed and (np.abs(e[bad] - thr) <= 1e-3 * thr).all(), f"{bad.sum()} pixels stopped without meeting the rule"
    sched = _schedule(min_spp, max_spp)
    for k in range(1, len(sched)):
        m = spp == sched[k]
        if not m.any():
            continue
        prev = sched[k - 1]
        u_rgb, u_stat, _ = gsc.render(cam, hs.params(width=64, spp=prev, seed=3, flags=api.FLAG_STATS, stat_clamp=CLAMP), want_stat=True)
        ep = _rule_error(u_rgb, u_stat, np.full(spp.shape, prev))
        bad = m & (ep <= thr)
        assert bad.sum() <= near_allowed and (np.abs(ep[bad] - thr) <= 1e-3 * thr).all(), \
            f"{bad.sum()} pixels went on past {prev} samples although they met the rule"
    assert stopped.any() and (spp > min_spp).any()
    gsc.close()


def test_list_longer_than_one_tile(rt, gpu_ctx):
    """320 x 240 pixels stay active after round 0: the list spans a whole 65 536-slot tile and a partial one."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, _, _, st, uni = _adaptive_vs_uniform(api, gsc, hs, 320, 2, 4, 0.0, height=240)
    assert (spp == 4).all() and st.rays == uni[4][2].rays
    gsc.close()


def test_several_waves_per_round(rt, gpu_ctx):
    """4096 paths in flight: round 0 alone (64 x 64 pixels x 4 samples) needs four waves to start its paths."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, _, _, _, _ = _adaptive_vs_uniform(api, gsc, hs, 64, 4, 32, 1.0, pool_paths=4096)
    assert len(np.unique(spp)) >= 2
    gsc.close()


def test_black_images_converge_at_min_spp(rt, gpu_ctx):
    """max_depth 0 (ray_color returns black at once) and a world without light: zero sums, zero variance, one round."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    rgb, spp, rgb8, _, st = gsc.render_adaptive(hs.camera(), hs.params(width=32, spp=64, max_depth=0), 4, 0.5)
    assert (spp == 4).all() and not rgb.any() and not rgb8.any() and st.paths == 4 * spp.size
    gsc.close()
    hs = api.HostScene("two_spheres", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    p = hs.params(width=32, spp=64)
    p.background[:] = [0.0, 0.0, 0.0]
    rgb, spp, rgb8, _, st = gsc.render_adaptive(hs.camera(), p, 4, 0.5)
    assert (spp == 4).all() and not rgb.any() and not rgb8.any() and st.rays >= st.paths
    gsc.close()


def test_demo_driver_max_error(rt, gpu_ctx):
    """`rt1w_main cornel_box --width 64 --spp 64 --max-error 1` prints what render_adaptive gives with the same arguments
    (seed 0, min_spp 16).  Two runs may add a pixel's samples in another order; only a pixel within rounding of the
    threshold could then stop at another count."""
    api = rt.api
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "rt1w_main")
    r = subprocess.run([exe, "cornel_box", "--width", "64", "--spp", "64", "--max-error", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stderr.rstrip().endswith("Done")
    lines = r.stdout.split("\n")
    assert lines[0] == "P3" and lines[1] == "64 64" and lines[2] == "255"
    body = np.array([[int(v) for v in ln.split()] for ln in lines[3:] if ln], dtype=np.int64).reshape(64, 64, 3)
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, spp, rgb8, _, _ = gsc.render_adaptive(hs.camera(), hs.params(width=64, spp=64, seed=0), 16, 1.0)
    assert len(np.unique(spp)) >= 2
    assert (body != rgb8).any(axis=2).sum() <= 4
    gsc.close()


def test_argument_checks(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()

    def status(min_spp=4, max_error=1.0, **kw):
        try:
            gsc.render_adaptive(cam, hs.params(width=16, **kw), min_spp, max_error)
            return api.OK
        except api.Rt1wError as e:
            return e.status

    assert status(spp=16) == api.OK
    assert status(spp=16, min_spp=16) == api.OK  # one uniform round
    assert status(spp=16, sample_begin=1) == api.ERR_INVALID
    assert status(spp=16, min_spp=1) == api.ERR_INVALID
    assert status(spp=16, min_spp=17) == api.ERR_INVALID
    assert status(spp=16, max_error=-0.5) == api.ERR_INVALID
    assert status(spp=16, max_error=float("nan")) == api.ERR_INVALID
    assert status(spp=1 << 24) == api.ERR_UNSUPPORTED
    gsc.close()


def test_multi_device_context_is_refused(rt, gpu_ctx):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    ctx = api.Context([0, 1])
    sc = api.Scene(ctx, hs.desc)
    with pytest.raises(api.Rt1wError) as e:
        sc.render_adaptive(hs.camera(), hs.params(width=16, spp=16), 4, 1.0)
    assert e.value.status == api.ERR_UNSUPPORTED and "one device" in str(e.value)
    sc.close(), ctx.close()
