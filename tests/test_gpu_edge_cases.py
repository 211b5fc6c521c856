"""Edge cases of the render entry points: smallest and largest images, ragged sizes, argument validation, seeds."""
import numpy as np
import pytest

from common import check_identical_render

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cornell(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    yield api, hs, gsc
    gsc.close()


def test_one_pixel_image(cornell):
    api, hs, gsc = cornell
    img, _, st = gsc.render(hs.camera(), hs.params(width=1, height=1, spp=3))
    assert img.shape == (1, 1, 3) and st.paths == 3 and st.rays >= 3
    assert np.isfinite(img).all()


def test_ragged_sizes_and_tiny_pools(cornell):
    """Odd image sizes and a wave capacity that divides nothing: scheduling changes, the estimate does not."""
    api, hs, gsc = cornell
    cam = hs.camera()
    ref = gsc.render(cam, hs.params(width=37, height=23, spp=5, seed=4))
    assert ref[0].shape == (23, 37, 3) and ref[2].paths == 37 * 23 * 5
    for pool in (257, 1025):
        got = gsc.render(cam, hs.params(width=37, height=23, spp=5, seed=4, pool_paths=pool))
        assert got[2].waves >= ref[2].waves
        check_identical_render(got, ref, f"pool {pool}", 5)


def test_largest_config_image(cornell):
    """BASELINE config 4's image size (3840x2160) with one sample: every path is started and accounted for."""
    api, hs, gsc = cornell
    p = hs.params(width=3840, height=2160, spp=1, max_depth=4)
    cam = hs.camera(aspect=3840 / 2160)
    img, _, st = gsc.render(cam, p)
    assert st.paths == 3840 * 2160 and st.rays >= st.paths and st.rays <= 4 * st.paths
    assert img.shape == (2160, 3840, 3) and np.isfinite(img).all() and img.max() > 0


def test_argument_validation(cornell):
    api, hs, gsc = cornell
    cam = hs.camera()
    for bad, status in ((dict(width=0), api.ERR_INVALID), (dict(spp=0), api.ERR_INVALID), (dict(spp=4, sample_begin=4), api.ERR_INVALID),
                        (dict(max_depth=256), api.ERR_UNSUPPORTED), (dict(sample_begin=-1, spp=3), api.ERR_INVALID)):
        kw = dict(width=8, spp=2)
        kw.update(bad)
        with pytest.raises(api.Rt1wError) as e:
            gsc.render(cam, hs.params(**kw))
        assert e.value.status == status, bad
    # max_depth = 255 is the last accepted value
    _, _, st = gsc.render(cam, hs.params(width=8, spp=1, max_depth=255))
    assert st.paths == 64


def test_seed_changes_the_stream_only(cornell):
    """Another seed: another Philox key, same estimator (image means agree within their noise)."""
    api, hs, gsc = cornell
    cam = hs.camera()
    a, _, _ = gsc.render(cam, hs.params(width=48, spp=64, seed=1))
    b, _, _ = gsc.render(cam, hs.params(width=48, spp=64, seed=2))
    c, _, _ = gsc.render(cam, hs.params(width=48, spp=64, seed=2 + (1 << 40)))  # the high seed word reaches the counter
    assert not np.array_equal(a, b) and not np.array_equal(b, c)
    ma, mb, mc = (np.nan_to_num(x).mean() for x in (a, b, c))
    assert abs(ma - mb) < 0.05 * ma and abs(mb - mc) < 0.05 * mb


def test_black_world_without_lights(rt, gpu_ctx):
    """No emitter and a black background: every path returns exactly zero (main.rs:113-115), rays are still traced."""
    api = rt.api
    hs = api.HostScene("two_spheres", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    p = hs.params(width=32, spp=4)
    p.background[:] = [0.0, 0.0, 0.0]
    img, _, st = gsc.render(hs.camera(), p)
    assert not img.any() and st.rays >= st.paths
    gsc.close()
