"""Converged-image parity (north_star check 3): CUDA wavefront renderer vs the f64 oracle.

The two sides use different RNG streams (Philox vs ChaCha12), so the comparison is statistical:
  * per pixel and channel, |mean_gpu - mean_oracle| <= 5 sigma of the difference for >= 99.9 % of them
    (means and variances of the per-sample radiance clamped at STAT_CLAMP on both sides);
  * the RMSE between the GPU image and an oracle image must not exceed the RMSE between two
    independent oracle images of the same sample count by more than 15 % (a bias would add to it);
  * whole-image mean radiance within 2 %.
"""
import numpy as np
import pytest

from common import check_identical_render, check_identical_sums, check_same_render, quantise

pytestmark = pytest.mark.gpu

STAT_CLAMP = 20.0

CASES = [
    # scene, width, spp
    ("cornel_box", 64, 512),
    ("cornel_smoke", 48, 256),
    ("random_scene", 96, 128),
    ("simple_light", 96, 256),
    ("two_perlin_spheres", 96, 128),
    ("earth", 96, 128),
    ("final_scene", 64, 256),
]


def _stats(stat, n):
    mean = stat[..., :3] / n
    var = np.maximum(stat[..., 3:] / n - mean * mean, 0.0)
    return mean, var


@pytest.mark.parametrize("name,width,spp", CASES)
def test_render_matches_oracle(rt, oracle, gpu_ctx, name, width, spp):
    api = rt.api
    hs = api.HostScene(name, seed=1)
    osc = oracle.OracleScene(hs.desc)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    p = hs.params(width=width, spp=spp, flags=api.FLAG_STATS, stat_clamp=STAT_CLAMP, seed=3)
    g_sum, g_stat, g_st = gsc.render(cam, p, want_stat=True)
    assert g_st.paths == p.width * p.height * spp
    oa_sum, oa_stat, oa_st = osc.render(cam, p, want_stat=True)
    pb = hs.params(width=width, spp=2 * spp, sample_begin=spp, flags=api.FLAG_STATS, stat_clamp=STAT_CLAMP)
    ob_sum, ob_stat, _ = osc.render(cam, pb, want_stat=True)

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

    assert abs(gm.mean() - am.mean()) <= 0.02 * am.mean() + 1e-4
    # rays per path agree too (same termination statistics)
    rpp_g, rpp_o = g_st.rays / g_st.paths, oa_st.rays / oa_st.paths
    assert abs(rpp_g - rpp_o) <= 0.02 * rpp_o, f"rays/path gpu {rpp_g:.3f} oracle {rpp_o:.3f}"
    gsc.close()


def test_sample_ranges_add_up(rt, gpu_ctx):
    """Sharding by sample range (the multi-GPU split) reproduces the single-call image up to fp32 summation order, ray for ray."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    full = gsc.render(cam, hs.params(width=48, spp=32, seed=9))
    a = gsc.render(cam, hs.params(width=48, spp=16, seed=9))
    b = gsc.render(cam, hs.params(width=48, spp=32, sample_begin=16, seed=9))
    assert a[2].rays + b[2].rays == full[2].rays and a[2].paths + b[2].paths == full[2].paths
    check_identical_sums(a[0] + b[0], full[0], 32, "[0, 16) + [16, 32)")
    # and a different pool size changes scheduling only, not the estimate
    c = gsc.render(cam, hs.params(width=48, spp=32, seed=9, pool_paths=4096))
    check_identical_render(c, full, "pool 4096", 32)
    gsc.close()


def test_depth_limits(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    img0, _, st0 = gsc.render(cam, hs.params(width=32, spp=4, max_depth=0))
    assert st0.rays == 0 and not img0.any()
    img1, _, st1 = gsc.render(cam, hs.params(width=32, spp=4, max_depth=1))
    assert st1.rays == 32 * 32 * 4  # exactly one closest-hit query per path
    assert img1.max() == pytest.approx(4 * 15.0)  # only directly visible light (emit 15, main.rs:414-418)
    gsc.close()


@pytest.mark.parametrize("name", ["random_scene", "final_scene"])
def test_bvh_wave_kernels_agree(rt, gpu_ctx, name):
    """The two wave kernels of BVH scenes (lockstep warps / lanes that take a new ray as soon as theirs is done) find the
    same closest hits and draw the same Philox numbers: the same image (common.check_same_render), ray for ray at depth 3."""
    api = rt.api
    hs = api.HostScene(name, seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    a = gsc.render(cam, hs.params(width=96, spp=16, seed=5, flags=api.FLAG_BVH_LOCKSTEP))
    b = gsc.render(cam, hs.params(width=96, spp=16, seed=5, flags=api.FLAG_BVH_PERSISTENT))
    check_same_render(a, b, name)
    a1 = gsc.render(cam, hs.params(width=96, spp=16, seed=5, flags=api.FLAG_BVH_LOCKSTEP, max_depth=3))  # shallow paths: no room to diverge
    b1 = gsc.render(cam, hs.params(width=96, spp=16, seed=5, flags=api.FLAG_BVH_PERSISTENT, max_depth=3))
    assert a1[2].rays == b1[2].rays
    gsc.close()


@pytest.mark.parametrize("name,width,spp", [("cornel_box", 128, 16), ("cornel_smoke", 96, 16), ("random_scene", 128, 8), ("final_scene", 64, 8),
                                            ("one_weekend", 128, 8), ("random_scene", 256, 1)])
def test_tail_kernel_changes_nothing(rt, gpu_ctx, name, width, spp):
    """The end of a render - once about one hit per resident thread is queued, ONE kernel follows every remaining path to
    its end inside a thread (render.cu: k_tail) instead of ~45 sparse waves - is the same computation: same scatter, same
    closest hit, same Philox counters.  With `RT1W_FLAG_NO_TAIL` (waves to the end) the same image, in fewer launches: the same
    rays, and the same sums up to the order of the fp32 additions (bit for bit at one sample per pixel)."""
    api = rt.api
    hs = api.HostScene(name, seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    a = gsc.render(cam, hs.params(width=width, spp=spp, seed=7))
    b = gsc.render(cam, hs.params(width=width, spp=spp, seed=7, flags=api.FLAG_NO_TAIL))
    check_identical_render(a, b, name, spp)
    assert a[2].waves < b[2].waves  # the tail kernel took over before depth 50
    c = gsc.render(cam, hs.params(width=width, spp=spp, seed=7, pool_paths=4096))  # many small waves, the tail kernel right away
    check_identical_render(a, c, name + ", small pool", spp)
    gsc.close()


@pytest.mark.parametrize("name,kw,width,spp,layout", [("random_scene", {}, 128, 8, "binary"), ("final_scene", {}, 64, 8, "wide"),
                                                      ("stress", dict(stress_spheres=100_000), 160, 8, None)])
def test_tail_kernel_of_the_persistent_scenes(rt, gpu_ctx, name, kw, width, spp, layout):
    """Scenes of the persistent wave kernel (k_wave_bvh: big trees, or forced) end the same way: k_tail on the tree and with the
    sine that kernel uses (render.cu: k_tail<.., WIDE, FAST_SIN = false>) - the same image as waves to the end."""
    api = rt.api
    hs = api.HostScene(name, seed=1, **kw)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    flags = api.FLAG_BVH_PERSISTENT | {"binary": api.FLAG_BVH_BINARY, "wide": api.FLAG_BVH_WIDE, None: 0}[layout]
    a = gsc.render(cam, hs.params(width=width, spp=spp, seed=7, flags=flags))
    b = gsc.render(cam, hs.params(width=width, spp=spp, seed=7, flags=flags | api.FLAG_NO_TAIL))
    check_identical_render(a, b, f"{name}, persistent kernel, {layout or 'default'} tree", spp)
    assert a[2].waves < b[2].waves  # the tail kernel took over before depth 50
    c = gsc.render(cam, hs.params(width=width, spp=spp, seed=7, flags=flags, pool_paths=4096))
    check_identical_render(a, c, name + ", persistent kernel, small pool", spp)
    gsc.close()

