"""BASELINE config 1 at FULL size (600x600, 100 spp, depth 50) on the GPU, checked through what does not need a
CPU render of that size: the reference's own published image, and size-independent properties of the estimator."""
import json
import os

import numpy as np
import pytest

from common import check_identical_sums
from test_oracle_golden_image import _linear_image, check_against_reference_png, load_golden

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def full(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(gpu_ctx, hs.desc)
    p = hs.params()  # the arm's own settings: 600 x 600, 100 spp, depth 50 (main.rs:867-894)
    assert (p.width, p.height, p.sample_end, p.max_depth) == (600, 600, 100, 50)
    img, _, st = gsc.render(hs.camera(), p)
    yield api, hs, gsc, img, st
    gsc.close()


def test_render_matches_reference_png(full):
    """The product against the reference's only published result (rest_of_your_life.png): the oracle's own bars - region
    means within 4 sqrt(2) sigma of a 100-spp realisation (about 0.5 %), the black frame, the share of pure-black pixels,
    the saturated light (tests/test_oracle_golden_image.py)."""
    api, hs, gsc, img, st = full
    assert st.paths == 600 * 600 * 100 and 4.9 < st.rays / st.paths < 5.3
    check_against_reference_png(_linear_image(img, 100), load_golden(), "gpu")


def test_eight_sample_ranges_add_up_at_full_size(full):
    """The multi-GPU split of config 4 (sample ranges, one per rank) at config 1's size: 8 shards == 1 render."""
    api, hs, gsc, img, st = full
    cam = hs.camera()
    total = np.zeros_like(img)
    rays = 0
    for r in range(8):
        s0, s1 = (100 * r) // 8, (100 * (r + 1)) // 8
        part, _, ps = gsc.render(cam, hs.params(spp=s1, sample_begin=s0))
        total += part
        rays += ps.rays
    assert rays == st.rays
    check_identical_sums(total, img, 100, "8 shards against one render")


def test_device_image_is_the_resolved_render(full):
    """rt1w_render_rgb8 at full size against the host resolve of the fp32 sums (summation order may move a level)."""
    api, hs, gsc, img, st = full
    rgb8, _ = gsc.render_rgb8(hs.camera(), hs.params())
    want = api.resolve_rgb8(img, 100).astype(np.int64)
    assert (np.abs(rgb8.astype(np.int64) - want) <= 1).mean() >= 0.9999
