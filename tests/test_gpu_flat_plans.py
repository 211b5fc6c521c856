"""Scan plans (csrc/flat_plans.h): a flat scene whose layout of scan groups matches a compiled plan is rendered by wave and
tail kernels with that layout unrolled at compile time; every other scene keeps the generic scan of the group table.

  * the shipped scenes report the plan they commit with (rt1w_scene_info.flat_plan);
  * a Cornell box with the light, the box and the sphere moved keeps plan 0, and its image renders (planned scan) equal the
    frame of a batch render (always the generic scan) bit for bit at one sample per pixel, samples 0 .. 7;
  * Cornell variants with another layout (no sphere, an unrotated box) get no plan and render as their batch frame too.
"""
import pytest

from common import check_identical_sums

pytestmark = pytest.mark.gpu

SPP = 8
SEED = 3
WIDTH = 400


def cornell(api, light=(213.0, 343.0, 227.0, 332.0), box_at=(265.0, 0.0, 295.0), box_deg=15.0, sphere=(190.0, 90.0, 190.0)):
    """The reference's cornel_box (main.rs:451-507) with the light, the box and the sphere where the arguments put them.
    box_deg None: the box without wrappers, at box_at; sphere None: no sphere."""
    b = api.DescBuilder()
    red, white, green = (b.lambertian(b.solid(*c)) for c in ((0.65, 0.05, 0.05), (0.73, 0.73, 0.73), (0.12, 0.45, 0.15)))
    lamp = b.diffuse_light(b.solid(15.0, 15.0, 15.0))
    aluminium = b.metal((0.8, 0.85, 0.88), 0.0)
    kids = [b.yz_rect(0, 555, 0, 555, 555, green), b.yz_rect(0, 555, 0, 555, 0, red),
            b.flip_face(b.xz_rect(*light, 554.0, lamp)),
            b.xz_rect(0, 555, 0, 555, 0, white), b.xz_rect(0, 555, 0, 555, 555, white), b.xy_rect(0, 555, 0, 555, 555, white)]
    if box_deg is None:
        kids.append(b.aabox(box_at, (box_at[0] + 165.0, box_at[1] + 330.0, box_at[2] + 165.0), aluminium))
    else:
        kids.append(b.translate(b.rotate_y(b.aabox((0.0, 0.0, 0.0), (165.0, 330.0, 165.0), aluminium), box_deg), box_at))
    lights = [b.xz_rect(*light, 554.0, b.null_material())]
    if sphere is not None:
        kids.append(b.sphere(sphere, 90.0, b.dielectric(1.5)))
        lights.append(b.sphere(sphere, 90.0, b.null_material()))
    b.set_world(b.bvh(kids))
    b.set_lights(lights)
    return b


def params(api, s0, n):
    p = api.RenderParams()
    p.width = p.height = WIDTH
    p.sample_begin, p.sample_end, p.max_depth, p.seed = s0, s0 + n, 50, SEED
    p.background[:] = [0.0, 0.0, 0.0]
    return p


def camera(api):
    return api.camera_new((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), (0.0, 1.0, 0.0), 40.0, 1.0, 0.0, 10.0, 0.0, 1.0)


@pytest.mark.parametrize("name,plan", [("cornel_box", 0), ("cornel_smoke", -1), ("two_spheres", -1), ("simple_light", -1)])
def test_shipped_scenes_report_their_plan(rt, gpu_ctx, name, plan):
    hs = rt.api.HostScene(name, seed=1)
    sc = rt.api.Scene(gpu_ctx, hs.desc)
    try:
        assert sc.info().flat_plan == plan
    finally:
        sc.close()


VARIANTS = {  # id: cornell() arguments, the plan the scene commits with
    "moved": (dict(light=(113.0, 443.0, 127.0, 432.0), box_at=(300.0, 0.0, 250.0), box_deg=-10.0, sphere=(400.0, 90.0, 120.0)), 0),
    "no_sphere": (dict(sphere=None), -1),
    "unrotated_box": (dict(box_deg=None, box_at=(300.0, 0.0, 250.0)), -1),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_variant_renders_as_its_batch_frame(rt, gpu_ctx, variant):
    """The image render (planned when the scene has a plan) against frame 0 of a one-frame batch (the generic scan) over the
    same paths: one sample per pixel, bit for bit, and the same rays."""
    api = rt.api
    kw, plan = VARIANTS[variant]
    b = cornell(api, **kw)
    sc = api.Scene(gpu_ctx, b.desc())
    try:
        info = sc.info()
        assert info.n_wide_nodes == 0 and info.n_prims <= 32, "the variant must be a flat-scan scene"
        assert info.flat_plan == plan
        cam = camera(api)
        for s0 in range(SPP):
            img, _, st = sc.render(cam, params(api, s0, 1))
            rgb, _, bst = sc.render_batch([cam], params(api, s0, 1), [SEED])
            check_identical_sums(img, rgb[0], 1, f"{variant}, sample {s0}", s0)
            assert st.paths == bst.paths and st.rays == bst.rays, f"{variant}, sample {s0}: {st.rays} rays against {bst.rays}"
        assert float(img.sum()) > 0.0
    finally:
        sc.close()
