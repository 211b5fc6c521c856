"""Schedule invariance: a path's random numbers depend only on its pixel, its sample index and the seed, so the image must not
depend on how the paths are scheduled - when the tail kernel (render.cu: k_tail) takes over, how many paths a wave holds, how
the sample range is split, whether the image is a frame of a batch, how many devices render it.

Every cell of scenes x schedules is compared with common.check_identical_render against the same render with waves to the end
(`RT1W_FLAG_NO_TAIL`) at the default wave capacity: eight one-sample renders (samples 0 .. 7), bit for bit - one path per pixel
and render, so a mismatch names the path - and one 8-sample render, up to the order of the fp32 additions.  The sizes are the
ones users render (random_scene 1200x800: 7.7 M paths and about 25 M rays per cell), so that a path that goes another way
once in 10^7 is seen.  The scenes run every kernel family: the flat scan with and without media (and the flat kernels' light
shortcut), the lockstep BVH kernel with solid colours and with media and rich textures, the persistent kernel on the binary
and the 8-wide tree."""
import numpy as np
import pytest

from common import check_identical_render, check_identical_sums

pytestmark = pytest.mark.gpu

SPP = 8
SEED = 5
STAT_CLAMP = 20.0

SCENES = {  # id: scene, constructor arguments, width, height (None: the arm's own), forced kernel
    "cornel_box": ("cornel_box", {}, 600, 600, None),
    "cornel_smoke": ("cornel_smoke", {}, 600, 600, None),
    "one_weekend": ("one_weekend", {}, None, None, None),
    "random_scene": ("random_scene", {}, 1200, 800, None),
    "final_scene": ("final_scene", {}, 800, 800, None),
    "random_scene-persistent-binary": ("random_scene", {}, 1200, 800, "persistent_binary"),
    "random_scene-persistent-wide": ("random_scene", {}, 1200, 800, "persistent_wide"),
    "stress": ("stress", dict(stress_spheres=200_000), None, None, None),
}

SCHEDULES = ["default", "tail_factor_0.25", "tail_factor_4", "tail_factor_64", "pool_65536", "pool_4096", "sample_split", "batch",
             "two_devices"]


class Cell:
    """One scene on the device, its renders with waves to the end (the references) and a way to render it again."""

    def __init__(self, api, ctx, sid):
        name, kw, width, height, kernel = SCENES[sid]
        self.api, self.sid = api, sid
        self.hs = api.HostScene(name, seed=1, **kw)
        s = self.hs.settings
        self.width, self.height = width or s.image_width, height or s.image_height
        self.flags = {None: 0, "persistent_binary": api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_BINARY,
                      "persistent_wide": api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_WIDE}[kernel]
        self.cam = self.hs.camera()
        self.gsc = api.Scene(ctx, self.hs.desc)
        self.ref1 = [self.render(self.gsc, s0, 1, no_tail=True) for s0 in range(SPP)]
        self.ref8 = self.render(self.gsc, 0, SPP, no_tail=True)

    def params(self, s0, n, no_tail=False, pool=0, stats=True, seed=SEED):
        flags = self.flags | (self.api.FLAG_NO_TAIL if no_tail else 0) | (self.api.FLAG_STATS if stats else 0)
        return self.hs.params(width=self.width, height=self.height, sample_begin=s0, sample_end=s0 + n, seed=seed, flags=flags,
                              stat_clamp=STAT_CLAMP, pool_paths=pool)

    def render(self, gsc, s0, n, no_tail=False, pool=0):
        return gsc.render(self.cam, self.params(s0, n, no_tail, pool), want_stat=True)

    def close(self):
        self.gsc.close()


@pytest.fixture(scope="module", params=list(SCENES))
def cell(request, rt, gpu_ctx):
    c = Cell(rt.api, gpu_ctx, request.param)
    rays = sum(r[2].rays for r in c.ref1) + c.ref8[2].rays
    print(f"[schedule invariance] {c.sid} {c.width}x{c.height}: {c.ref8[2].paths} paths, {rays} rays per cell")
    yield c
    c.close()


def _same_schedule_renders(c, gsc, label, pool=0):
    """The eight one-sample renders and the 8-sample render of `gsc` against the references."""
    for s0 in range(SPP):
        check_identical_render(c.render(gsc, s0, 1, pool=pool), c.ref1[s0], f"{label}, sample {s0}", 1, s0)
    got = c.render(gsc, 0, SPP, pool=pool)
    check_identical_render(got, c.ref8, f"{label}, {SPP} spp", SPP)
    return got


@pytest.mark.parametrize("schedule", SCHEDULES)
def test_schedule_changes_nothing(rt, gpu_ctx, cell, schedule, monkeypatch):
    api, c = rt.api, cell
    label = f"{c.sid} {c.width}x{c.height}, {schedule}"
    if schedule == "default":
        _same_schedule_renders(c, c.gsc, label)
    elif schedule.startswith("tail_factor_"):  # render_waves reads RT1W_TAIL_FACTOR on every render
        monkeypatch.setenv("RT1W_TAIL_FACTOR", schedule[len("tail_factor_"):])
        _same_schedule_renders(c, c.gsc, label)
    elif schedule.startswith("pool_"):
        _same_schedule_renders(c, c.gsc, label, pool=int(schedule[len("pool_"):]))
    elif schedule == "sample_split":  # [0, 4) + [4, 8) against [0, 8)
        lo, hi = c.render(c.gsc, 0, SPP // 2), c.render(c.gsc, SPP // 2, SPP // 2)
        assert lo[2].paths + hi[2].paths == c.ref8[2].paths
        assert lo[2].rays + hi[2].rays == c.ref8[2].rays, f"{label}: {lo[2].rays} + {hi[2].rays} rays against {c.ref8[2].rays}"
        check_identical_sums(lo[0] + hi[0], c.ref8[0], SPP, label)
        check_identical_sums(lo[1] + hi[1], c.ref8[1], SPP, label + " (statistics)")
    elif schedule == "batch":  # frame 0 with the references' seed, frame 1 with another one; tiles straddle the frames
        for s0, n in [(s0, 1) for s0 in range(SPP)] + [(0, SPP)]:
            rgb, _, st = c.gsc.render_batch([c.cam, c.cam], c.params(s0, n, stats=False), [SEED, SEED + 1])
            other = c.gsc.render(c.cam, c.params(s0, n, no_tail=True, stats=False, seed=SEED + 1))
            ref = c.ref1[s0] if n == 1 else c.ref8
            check_identical_sums(rgb[0], ref[0], n, f"{label}, frame 0, samples [{s0}, {s0 + n})", s0)
            check_identical_sums(rgb[1], other[0], n, f"{label}, frame 1, samples [{s0}, {s0 + n})", s0)
            assert st.paths == ref[2].paths + other[2].paths
            assert st.rays == ref[2].rays + other[2].rays, f"{label}, samples [{s0}, {s0 + n}): {st.rays} rays against {ref[2].rays} + {other[2].rays}"
    elif schedule == "two_devices":  # the sample range sharded over two devices, the sums added by ncclReduce
        import torch

        if torch.cuda.device_count() < 2:
            pytest.skip("needs 2 GPUs")
        ctx2 = api.Context([0, 1])
        gsc2 = api.Scene(ctx2, c.hs.desc)
        try:
            _same_schedule_renders(c, gsc2, label)
        finally:
            gsc2.close(), ctx2.close()
    else:
        raise AssertionError(schedule)
