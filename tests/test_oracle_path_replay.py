"""The oracle's path replay (oracle.h: oracle_replay_paths) on the CPU: its camera rays against a numpy restatement of the
device's camera_ray driven by rt1w_philox4x32, its depth-1 radiance, and its determinism.  (The replay against the device
render is tests/test_gpu_path_replay.py.)"""
import numpy as np
import pytest

from common import pixel_seeds

SEED_HI = 0x9E3779B9_00000005


def u01(x):
    return np.float32(np.uint32(x) >> np.uint32(8)) * np.float32(1.0 / 16777216.0)


def camera_ray(api, cam, w, h, pix, s, seed):
    """render.cu: camera_ray - counter (s, 0, RNG_CAMERA ^ (seed hi << 4), block), key (pixel seed, seed lo)."""
    key = (pix, seed & 0xFFFFFFFF)
    word = 0 ^ ((seed >> 32) << 4)
    x = api.philox4x32((s, 0, word, 0), key)
    j, i = pix // w, pix % w
    ss = (i + float(u01(x[0]))) / (w - 1)
    tt = (j + float(u01(x[1]))) / (h - 1)
    off = np.zeros(3)
    if cam.lens_radius != 0.0:
        b = 1
        while True:
            y = api.philox4x32((s, 0, word, b), key)
            b += 1
            px, py = np.float32(2) * u01(y[0]) - np.float32(1), np.float32(2) * u01(y[1]) - np.float32(1)
            if px * px + py * py < np.float32(1):
                break
            px, py = np.float32(2) * u01(y[2]) - np.float32(1), np.float32(2) * u01(y[3]) - np.float32(1)
            if px * px + py * py < np.float32(1):
                break
        off = np.array(cam.u[:]) * (cam.lens_radius * float(px)) + np.array(cam.v[:]) * (cam.lens_radius * float(py))
    o = np.array(cam.origin[:])
    d = np.array(cam.lower_left_corner[:]) + ss * np.array(cam.horizontal[:]) + tt * np.array(cam.vertical[:]) - o - off
    time = np.float32(cam.time0 + (cam.time1 - cam.time0) * float(u01(x[2])))
    return o + off, d.astype(np.float32), time


@pytest.mark.parametrize("name", ["cornel_box", "random_scene"])  # pinhole; lens and shutter
@pytest.mark.parametrize("seed", [0, SEED_HI])
def test_camera_rays_follow_the_draw_map(rt, oracle, name, seed):
    api = rt.api
    hs = api.HostScene(name, seed=1)
    osc = oracle.OracleScene(hs.desc)
    cam = hs.camera()
    assert (cam.lens_radius != 0.0) == (name == "random_scene")
    p = hs.params(width=40, sample_begin=0, sample_end=1, seed=seed)
    rng = np.random.default_rng(5)
    pix = rng.integers(0, p.width * p.height, 48).astype(np.uint32)
    samples = rng.choice([0, 5, 65539, 1 << 20], 48).astype(np.int32)
    o, d, t = osc.replay_camera_rays(cam, p, pix, samples)
    for k in range(48):
        wo, wd, wt = camera_ray(api, cam, p.width, p.height, int(pix[k]), int(samples[k]), seed)
        np.testing.assert_allclose(o[k], wo, rtol=1e-14, atol=1e-12)
        # f32 directions: the same value, or one ulp apart where the f64 sums round on either side of a half-ulp
        assert np.all(np.abs(d[k] - wd.astype(np.float64)) <= np.spacing(np.abs(wd)).astype(np.float64)), (k, d[k], wd)
        assert t[k] == float(wt)
    # swapping the jitters (mutation 9) moves the rays: the restatement above is not vacuous
    _, d9, _ = osc.replay_camera_rays(cam, p, pix, samples, mutation=9)
    assert np.mean(np.any(d9 != d, axis=1)) > 0.9


@pytest.mark.parametrize("name", ["cornel_box", "simple_light", "cornel_smoke", "two_spheres"])
def test_depth_one_is_background_or_emission(rt, oracle, name):
    """At max_depth = 1 the throughput is 1: every path is its camera ray's background, the emission of the light it hits,
    0 on any other surface, or NaN where that surface's Lambertian pdf is 0 (main.rs:102)."""
    api = rt.api
    hs = api.HostScene(name, seed=1)
    osc = oracle.OracleScene(hs.desc)
    p = hs.params(width=48, sample_begin=0, sample_end=1, seed=SEED_HI, max_depth=1)
    seeds = pixel_seeds((p.height, p.width)).reshape(-1)
    rgb, rays, flags = osc.replay_paths(hs.camera(), p, seeds, np.zeros(seeds.size, np.int32), threads=2)
    assert (rays == 1).all()
    desc = hs.desc.contents
    allowed = [tuple(p.background[:]), (0.0, 0.0, 0.0)]
    for m in range(desc.n_materials):
        mat = desc.materials[m]
        if mat.type == api.MAT_DIFFUSE_LIGHT and desc.textures[mat.texture].type == api.TEX_SOLID:
            allowed.append(tuple(desc.textures[mat.texture].color[:]))
    allowed = np.array(allowed)
    fin = ~np.isnan(rgb).any(axis=1)
    ok = (rgb[fin][:, None, :] == allowed[None]).all(axis=2).any(axis=1)
    assert ok.all(), f"{name}: {np.sum(~ok)} depth-1 paths are neither background nor emission nor 0: {rgb[fin][~ok][:3]}"
    # both a light and a miss or a surface are seen, so the check is not vacuous
    assert len({tuple(x) for x in rgb[fin]}) >= 2


@pytest.mark.parametrize("name", ["cornel_smoke", "random_scene"])
def test_replay_is_deterministic_across_thread_counts(rt, oracle, name):
    api = rt.api
    hs = api.HostScene(name, seed=1)
    osc = oracle.OracleScene(hs.desc)
    p = hs.params(width=48, sample_begin=5, sample_end=6, seed=SEED_HI, max_depth=50)
    seeds = pixel_seeds((p.height, p.width)).reshape(-1)
    samples = np.full(seeds.size, 5, np.int32)
    lmap = np.arange(osc.num_prims, dtype=np.int32)
    a = osc.replay_paths(hs.camera(), p, seeds, samples, lmap, threads=1)
    b = osc.replay_paths(hs.camera(), p, seeds, samples, lmap, threads=4)
    assert np.array_equal(a[0].view(np.uint64), b[0].view(np.uint64))
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert a[1].sum() > seeds.size  # paths bounce


def test_every_mutation_changes_some_path(rt, oracle):
    """Each mutation (oracle.h) changes some replayed path of the scene built to show it: the device comparison in
    test_gpu_path_replay.py can only catch what the replay distinguishes."""
    api = rt.api
    hs = api.HostScene("random_scene", seed=1)
    osc = oracle.OracleScene(hs.desc)
    p = hs.params(width=64, sample_begin=5, sample_end=6, seed=SEED_HI, max_depth=3)
    seeds = pixel_seeds((p.height, p.width)).reshape(-1)
    samples = np.full(seeds.size, 5, np.int32)
    base, _, _ = osc.replay_paths(hs.camera(), p, seeds, samples, threads=2)
    for mutation in (1, 2, 4, 7, 8, 9):
        mut, _, _ = osc.replay_paths(hs.camera(), p, seeds, samples, mutation=mutation, threads=2)
        differ = ~((mut == base) | (np.isnan(mut) & np.isnan(base))).all(axis=1)
        assert differ.mean() > 0.01, f"mutation {mutation} changes only {differ.mean():.4f} of the paths"


def test_leaf_map_inverts_the_leaf_table(oracle):
    leaf_prims = np.array([3, 0, 2, 1], np.int32)
    assert oracle.replay_leaf_map(leaf_prims, 5).tolist() == [1, 3, 2, 0, -1]


def test_path_log_explains_a_path(rt, oracle):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    osc = oracle.OracleScene(hs.desc)
    p = hs.params(width=32, sample_begin=0, sample_end=1, seed=0, max_depth=50)
    text = osc.replay_path_log(hs.camera(), p, 32 * 16 + 16, 0)
    assert text.startswith("pixel seed 528 sample 0") and "depth 0: prim" in text
