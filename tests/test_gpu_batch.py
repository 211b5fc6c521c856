"""Batch rendering (include/rt1w.h: rt1w_render_batch).  Frame f of a batch keys Philox exactly as rt1w_render of its
camera and seed, so every frame must hold what that render gives - sums, NaNs and ray counts - up to the order of the fp32
additions.  Checked on every kernel family (flat scan, media, lockstep and persistent BVH kernels, binary and 8-wide trees,
the tail kernel and its absence), on the path numbering's edge cases (tiles that straddle frames, small pools, many tiny
frames), on seeds and sample ranges, on the argument checks, on a two-device context and through the demo driver."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _same_sums(a, b, label):
    assert (np.isnan(a) == np.isnan(b)).all(), f"{label}: NaN in different places"
    ok = ~np.isnan(a)
    np.testing.assert_allclose(a[ok], b[ok], rtol=1e-4, atol=1e-4, err_msg=label)


def _cameras(api, hs, n=3):
    """n views of the scene: the scene's own camera, then look_from turned about the vertical axis through look_at and pulled
    in, with a lens (aperture 0.1 .. ) and shutter windows of their own (moving spheres move between them)."""
    s = hs.settings
    lf, la = np.array(s.look_from[:]), np.array(s.look_at[:])
    cams = [hs.camera()]
    for k in range(1, n):
        a = math.radians(25.0 * k)
        arm = (lf - la) * (1.0 - 0.1 * k)
        turned = la + np.array([math.cos(a) * arm[0] + math.sin(a) * arm[2], arm[1], -math.sin(a) * arm[0] + math.cos(a) * arm[2]])
        t0 = 0.2 * (k % 3)
        cams.append(api.camera_new(turned.tolist(), la.tolist(), [0.0, 1.0, 0.0], s.vfov_deg, s.aspect_ratio, 0.1 * (k % 2) + s.aperture, 10.0,
                                   t0, t0 + 0.3))
    return cams


def _batch_vs_singles(api, gsc, cams, params, seeds, label):
    """The batch, then every frame's single render: sums, device resolve, rays and paths.  -> (rgb_sum, rgb8, stats)."""
    rgb, rgb8, st = gsc.render_batch(cams, params, seeds)
    n, h, w = len(cams), params.height, params.width
    assert rgb.shape == (n, h, w, 3) and rgb8.shape == (n, h, w, 3)
    spp = params.sample_end - params.sample_begin
    rays = paths = 0
    for f, cam in enumerate(cams):
        p = api.RenderParams.from_buffer_copy(params)
        p.seed = int(seeds[f]) if seeds is not None else params.seed
        ref, _, sst = gsc.render(cam, p)
        _same_sums(rgb[f], ref, f"{label}: frame {f}")
        assert np.array_equal(rgb8[f], api.resolve_rgb8(rgb[f], spp)), f"{label}: device resolve of frame {f}"
        rays, paths = rays + sst.rays, paths + sst.paths
    assert st.paths == paths == n * h * w * spp, label
    assert st.rays == rays, f"{label}: {st.rays} rays in the batch, {rays} in the single renders"
    return rgb, rgb8, st


CASES = [  # scene, constructor arguments, width, flags: flat scan, flat + media, lockstep binary tree (lens, moving spheres),
    # media + rich textures, persistent 8-wide tree, persistent binary tree, no tail kernel
    ("cornel_box", {}, 64, 0),
    ("cornel_smoke", {}, 64, 0),
    ("random_scene", {}, 96, 0),
    ("final_scene", {}, 64, 0),
    ("stress", dict(stress_spheres=200_000), 96, 0),
    ("random_scene", {}, 96, "persistent_binary"),
    ("cornel_smoke", {}, 64, "no_tail"),
]


@pytest.mark.parametrize("name,kw,width,flags", CASES, ids=[f"{c[0]}-{c[3] or 'default'}" for c in CASES])
def test_every_frame_equals_its_single_render(rt, gpu_ctx, name, kw, width, flags):
    api = rt.api
    flags = {"persistent_binary": api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_BINARY, "no_tail": api.FLAG_NO_TAIL}.get(flags, flags)
    hs = api.HostScene(name, seed=1, **kw)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cams = _cameras(api, hs)
    seeds = [11, 12, (5 << 32) | 13]  # the last one keys with a seed high word
    _, _, st = _batch_vs_singles(api, gsc, cams, hs.params(width=width, spp=8, flags=flags), seeds, name)
    print(f"[batch {name}] {st.paths} paths, {st.rays} rays, {st.waves} waves, {st.launches} launches, {st.render_ms:.2f} ms")
    gsc.close()


def test_tiles_straddle_frames(rt, gpu_ctx):
    """300 x 229 = 68 700 pixels per frame: the 65 536-pixel tiles of the path numbering start inside frames."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _batch_vs_singles(api, gsc, _cameras(api, hs), hs.params(width=300, height=229, spp=4), [1, 2, 3], "300x229")
    gsc.close()


def test_small_pool(rt, gpu_ctx):
    """4096 paths in flight: the frames' paths start over many waves."""
    api = rt.api
    hs = api.HostScene("cornel_smoke", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    _, _, st = _batch_vs_singles(api, gsc, _cameras(api, hs, 4), hs.params(width=32, spp=8, pool_paths=4096), [5, 6, 7, 8], "pool 4096")
    assert st.waves > 8
    gsc.close()


def test_many_tiny_frames(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cams = _cameras(api, hs, 4) * 50
    _batch_vs_singles(api, gsc, cams, hs.params(width=16, height=9, spp=4), list(range(200)), "200 frames of 16x9")
    gsc.close()


def test_seeds(rt, gpu_ctx):
    """seeds=None is params.seed for every frame; equal cameras and seeds give equal frames, other seeds other frames."""
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cam = hs.camera()
    p = hs.params(width=48, spp=8, seed=9)
    a, _, sa = gsc.render_batch([cam, cam, cam], p)
    b, _, sb = gsc.render_batch([cam, cam, cam], p, [9, 9, 9])
    _same_sums(a, b, "seeds=None against params.seed")
    assert sa.rays == sb.rays
    c, _, _ = gsc.render_batch([cam, cam, cam], p, [4, 4, 5])
    _same_sums(c[0], c[1], "two frames with one camera and seed")
    assert not np.allclose(c[0], c[2], equal_nan=True), "another seed should give another image"
    gsc.close()


def test_sample_ranges(rt, gpu_ctx):
    """One frame is rt1w_render (rays included); [0, 8) + [8, 16) of a batch add up to [0, 16)."""
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    cams = _cameras(api, hs)
    _batch_vs_singles(api, gsc, cams[1:2], hs.params(width=64, spp=8, seed=3), None, "one frame")
    lo, _, s_lo = gsc.render_batch(cams, hs.params(width=64, sample_begin=0, sample_end=8), [1, 2, 3])
    hi, _, s_hi = gsc.render_batch(cams, hs.params(width=64, sample_begin=8, sample_end=16), [1, 2, 3])
    whole, _, s_all = gsc.render_batch(cams, hs.params(width=64, spp=16), [1, 2, 3])
    _same_sums(lo + hi, whole, "[0, 8) + [8, 16)")
    assert s_lo.rays + s_hi.rays == s_all.rays and s_lo.paths + s_hi.paths == s_all.paths
    gsc.close()


def test_argument_checks(rt):
    import torch

    api = rt.api
    lib = api.load_library()
    ctx = api.Context(0)  # its own context: the 2^32-pixel call must not leave buffers behind
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    out, out8 = np.zeros(16 * 16 * 3 * 2, np.float32), np.zeros(16 * 16 * 3 * 2, np.uint8)

    def status(cams, n, params, rgb_sum=out.ctypes.data, rgb8=None):
        return lib.rt1w_render_batch(gsc._h, cams, n, None, C.byref(params), rgb_sum, rgb8, None)

    two = (api.Camera * 2)(cam, cam)
    p = hs.params(width=16, height=16, spp=4)
    assert status(two, 2, p) == api.OK
    assert status(two, 2, p, rgb_sum=None, rgb8=out8.ctypes.data) == api.OK
    assert status(two, 0, p) == api.ERR_INVALID
    assert status(two, -1, p) == api.ERR_INVALID
    assert status(None, 2, p) == api.ERR_INVALID
    assert status(two, 2, p, rgb_sum=None, rgb8=None) == api.ERR_INVALID
    assert status(two, 2, hs.params(width=16, height=16, spp=4, flags=api.FLAG_STATS)) == api.ERR_INVALID
    assert status(two, 2, hs.params(width=0, height=16, spp=4)) == api.ERR_INVALID
    assert status(two, 2, hs.params(width=16, height=16, sample_begin=4, sample_end=4)) == api.ERR_INVALID
    assert status(two, 2, hs.params(width=16, height=16, spp=1 << 24)) == api.ERR_UNSUPPORTED
    # exactly 2^32 batch pixels: refused before anything is allocated (its sums alone would take 48 GB)
    many = (api.Camera * 65536)(*([cam] * 65536))
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(0)
    assert status(many, 65536, hs.params(width=256, height=256, spp=1)) == api.ERR_INVALID
    free1, _ = torch.cuda.mem_get_info(0)
    assert free0 - free1 < (1 << 30), f"{(free0 - free1) / 2**30:.1f} GB allocated by a refused call"
    gsc.close(), ctx.close()


def test_two_device_context(rt, gpu_ctx):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    cams, p, seeds = _cameras(api, hs), hs.params(width=64, spp=8), [1, 2, 3]
    one = api.Scene(gpu_ctx, hs.desc)
    a, a8, sa = one.render_batch(cams, p, seeds)
    ctx2 = api.Context([0, 1])
    two = api.Scene(ctx2, hs.desc)
    b, b8, sb = two.render_batch(cams, p, seeds)
    _same_sums(a, b, "two devices against one")
    assert sa.rays == sb.rays and sa.paths == sb.paths
    assert np.array_equal(b8, np.stack([api.resolve_rgb8(b[f], 8) for f in range(len(cams))]))
    two.close(), ctx2.close(), one.close()


def _turntable_camera(api, hs, k, n):
    s = hs.settings
    lf, la = np.array(s.look_from[:]), np.array(s.look_at[:])
    a, arm = 2.0 * math.pi * k / n, lf - la
    eye = lf if k == 0 else la + np.array([math.cos(a) * arm[0] + math.sin(a) * arm[2], arm[1], -math.sin(a) * arm[0] + math.cos(a) * arm[2]])
    return api.camera_new(eye.tolist(), la.tolist(), [0.0, 1.0, 0.0], s.vfov_deg, s.aspect_ratio, s.aperture, 10.0, 0.0, 1.0)


def test_demo_driver_frames(rt, gpu_ctx):
    """`rt1w_main random_scene --width 48 --spp 8 --frames 3` prints three P3 images: frame k is the view turned by k * 120
    degrees about the vertical axis through look_at, rendered with seed k."""
    api = rt.api
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "rt1w_main")
    r = subprocess.run([exe, "random_scene", "--width", "48", "--spp", "8", "--frames", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stderr.rstrip().endswith("Done")
    hs = api.HostScene("random_scene", seed=1)
    w, h = 48, int(48 / hs.settings.aspect_ratio)
    lines = [ln for ln in r.stdout.split("\n") if ln]
    per = 3 + w * h
    assert len(lines) == 3 * per
    gsc = api.Scene(gpu_ctx, hs.desc)
    for k in range(3):
        head = lines[k * per: k * per + 3]
        assert head == ["P3", f"{w} {h}", "255"], head
        body = np.array([[int(v) for v in ln.split()] for ln in lines[k * per + 3: (k + 1) * per]], dtype=np.int64).reshape(h, w, 3)
        ref, _ = gsc.render_rgb8(_turntable_camera(api, hs, k, 3), hs.params(width=48, spp=8, seed=k))
        close = np.abs(body - ref.astype(np.int64)) <= 1
        assert close.mean() >= 0.999, f"frame {k}: {(~close).sum()} values differ by more than one level"
    gsc.close()
    r = subprocess.run([exe, "random_scene", "--width", "48", "--spp", "8", "--frames", "3", "--max-error", "1"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0
