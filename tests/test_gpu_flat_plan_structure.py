"""Plans cover the whole structure of a flat scene (csrc/flat_plans.h): besides the group layout of the scan, the primitive class
of every scan slot (pass 2), the op kinds of every wrapper chain (finalize_hit) and the kinds of the light list, in order
(scatter_lambertian).  A scene that differs in any of them commits without a plan and keeps the generic kernels.

  * a Cornell box with the light, the box, its angle and the sphere moved keeps plan 0, and its image renders (the planned
    kernels) equal the frame of a batch render (the generic kernels) bit for bit at one sample per pixel, samples 0 .. 7,
    with the same ray counts;
  * variants with the group layout of plan 0 but another light list (sphere first, a third light) or another wrapper chain
    (RotateY alone, a FlipFace in the chain) get no plan and render as their batch frame too.
"""
import pytest

from common import check_identical_sums

pytestmark = pytest.mark.gpu

SPP = 8
SEED = 5
WIDTH = 320


def cornell(api, light=(213.0, 343.0, 227.0, 332.0), box_at=(265.0, 0.0, 295.0), box_deg=15.0, sphere=(190.0, 90.0, 190.0),
            radius=90.0, chain="rotate_translate", lights="rect_sphere"):
    """The reference's cornel_box (main.rs:451-507) with the geometry the arguments give.
    chain: the wrappers of the box, innermost first - "rotate_translate" (the reference's), "rotate" (RotateY alone, the box
    at the origin), "flip_rotate_translate" (FlipFace, RotateY, Translate).
    lights: the light list - "rect_sphere" (the reference's), "sphere_rect", "rect_sphere_rect" (a second ceiling lamp)."""
    b = api.DescBuilder()
    red, white, green = (b.lambertian(b.solid(*c)) for c in ((0.65, 0.05, 0.05), (0.73, 0.73, 0.73), (0.12, 0.45, 0.15)))
    lamp = b.diffuse_light(b.solid(15.0, 15.0, 15.0))
    aluminium = b.metal((0.8, 0.85, 0.88), 0.0)
    kids = [b.yz_rect(0, 555, 0, 555, 555, green), b.yz_rect(0, 555, 0, 555, 0, red),
            b.flip_face(b.xz_rect(*light, 554.0, lamp)),
            b.xz_rect(0, 555, 0, 555, 0, white), b.xz_rect(0, 555, 0, 555, 555, white), b.xy_rect(0, 555, 0, 555, 555, white)]
    box = b.aabox((0.0, 0.0, 0.0), (165.0, 330.0, 165.0), aluminium)
    if chain == "rotate_translate":
        box = b.translate(b.rotate_y(box, box_deg), box_at)
    elif chain == "rotate":
        box = b.rotate_y(box, box_deg)
    elif chain == "flip_rotate_translate":
        box = b.translate(b.rotate_y(b.flip_face(box), box_deg), box_at)
    else:
        raise ValueError(chain)
    kids.append(box)
    kids.append(b.sphere(sphere, radius, b.dielectric(1.5)))
    b.set_world(b.bvh(kids))
    rect = b.xz_rect(*light, 554.0, b.null_material())
    ball = b.sphere(sphere, radius, b.null_material())
    b.set_lights({"rect_sphere": [rect, ball], "sphere_rect": [ball, rect],
                  "rect_sphere_rect": [rect, ball, b.xz_rect(100.0, 180.0, 100.0, 180.0, 554.0, b.null_material())]}[lights])
    return b


def params(api, s0, n):
    p = api.RenderParams()
    p.width = p.height = WIDTH
    p.sample_begin, p.sample_end, p.max_depth, p.seed = s0, s0 + n, 50, SEED
    p.background[:] = [0.0, 0.0, 0.0]
    return p


def camera(api):
    return api.camera_new((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), (0.0, 1.0, 0.0), 40.0, 1.0, 0.0, 10.0, 0.0, 1.0)


VARIANTS = {  # id: cornell() arguments, the plan the scene commits with
    "moved": (dict(light=(150.0, 400.0, 180.0, 300.0), box_at=(320.0, 0.0, 200.0), box_deg=33.0, sphere=(160.0, 120.0, 330.0),
                   radius=70.0), 0),
    "lights_sphere_first": (dict(lights="sphere_rect"), -1),
    "third_light": (dict(lights="rect_sphere_rect"), -1),
    "box_rotate_only": (dict(chain="rotate", box_deg=-20.0), -1),
    "box_flip_in_chain": (dict(chain="flip_rotate_translate"), -1),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_structure_variant_renders_as_its_batch_frame(rt, gpu_ctx, variant):
    """The image render (planned when the scene has a plan) against frame 0 of a one-frame batch (always the generic kernels)
    over the same paths: one sample per pixel, bit for bit, and the same rays."""
    api = rt.api
    kw, plan = VARIANTS[variant]
    sc = api.Scene(gpu_ctx, cornell(api, **kw).desc())
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
