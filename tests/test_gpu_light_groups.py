"""Light groups (include/rt1w.h: rt1w_render_light_groups).  A path's radiance comes from the one event that ends it, and
emission never steers a path, so the group render traces exactly rt1w_render's paths and rays and only splits the sums:
  * summed over the groups they are rt1w_render's sums (common.check_identical_render: bit for bit at 1 spp), on every
    kernel family - flat scan, media, rich textures, lockstep and persistent BVH kernels, binary and 8-wide trees, a global
    emitter under FlipFace, an emissive AABox in a tree, a light under Translate / RotateY;
  * group k is its light's share: the render of the scene with that light's emission (or the background) doubled is the
    relight with 2 on group k, bit for bit at 1 spp (x2 is exact in f32), and merged groups are the sums of their parts;
  * schedules (no tail kernel, small pools, sample ranges, two devices) move nothing;
  * the argument checks and the demo driver."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import check_identical_render, check_identical_sums
from test_gpu_adhoc_scenes import AdHoc, enclosed_scene

pytestmark = pytest.mark.gpu


def lights_scene(api):
    """An emissive AABox among 40 spheres inside a BVH (more than the flat scan's 32 primitives: the box is one P_BOX leaf of
    the tree) and a rectangle light under Translate / RotateY, over a floor, with a dim blue background."""
    rng = np.random.Generator(np.random.Philox(23))
    b = api.DescBuilder()
    grey, red = b.lambertian(b.solid(0.6, 0.6, 0.6)), b.lambertian(b.solid(0.7, 0.2, 0.2))
    kids = [b.xz_rect(-200.0, 200.0, -200.0, 200.0, 0.0, grey),
            b.aabox((-20.0, 0.0, -20.0), (20.0, 15.0, 20.0), b.diffuse_light(b.solid(4.0, 3.0, 2.0))),
            b.rotate_y(b.translate(b.xz_rect(-15.0, 15.0, -10.0, 10.0, 0.0, b.diffuse_light(b.solid(2.0, 5.0, 7.0))), (30.0, 60.0, 10.0)), 30.0),
            b.sphere((0.0, 30.0, 0.0), 12.0, b.metal((0.8, 0.8, 0.9), 0.05))]
    for k in range(40):
        c = rng.uniform(-90.0, 90.0, 3)
        c[1] = rng.uniform(4.0, 40.0)
        kids.append(b.sphere(tuple(c), float(rng.uniform(2.0, 6.0)), red if k % 3 else grey))
    b.set_world(b.bvh(kids))
    return AdHoc(api, b, (0.0, 80.0, -200.0), (0.0, 20.0, 0.0), 50.0, (0.05, 0.06, 0.1))


def _scene(api, name):
    """-> (host scene, camera, make_params(width, begin, end, flags, pool))."""
    if name == "enclosed":
        hs = enclosed_scene(api)
    elif name == "lights":
        hs = lights_scene(api)
    else:
        hs = api.HostScene(name, seed=1, **(dict(stress_spheres=200_000) if name == "stress" else {}))
    if isinstance(hs, AdHoc):
        def params(width, begin, end, flags=0, pool=0):
            p = hs.params(width, end, sample_begin=begin, flags=flags)
            p.pool_paths = pool
            return p
    else:
        def params(width, begin, end, flags=0, pool=0):
            return hs.params(width=width, sample_begin=begin, sample_end=end, flags=flags, pool_paths=pool)
    return hs, hs.camera(), params


def _relit_desc(api, desc, node=None, material=None, factor=2.0):
    """A copy of the description in which one light node gets a DiffuseLight of `factor` times its emission (node), or one
    DiffuseLight material emits `factor` times as much (material: every light that shares it).  Solid-colour emitters only."""
    d = desc.contents if isinstance(desc, C.POINTER(api.SceneDesc)) else desc
    nodes = (api.Node * d.n_nodes)(*d.nodes[: d.n_nodes])
    mats = (api.Material * (d.n_materials + 1))(*d.materials[: d.n_materials])
    texs = (api.Texture * (d.n_textures + 1))(*d.textures[: d.n_textures])
    m = nodes[node].material if node is not None else material
    assert mats[m].type == api.MAT_DIFFUSE_LIGHT and texs[mats[m].texture].type == api.TEX_SOLID
    t = api.Texture.from_buffer_copy(texs[mats[m].texture])
    t.color[:] = [factor * x for x in t.color]
    texs[d.n_textures] = t
    if node is not None:
        mats[d.n_materials] = api.Material.from_buffer_copy(mats[m])
        mats[d.n_materials].texture = d.n_textures
        nodes[node].material = d.n_materials
    else:
        mats[m].texture = d.n_textures
    out = api.SceneDesc.from_buffer_copy(d)
    out.nodes, out.materials, out.n_materials = nodes, mats, d.n_materials + 1
    out.textures, out.n_textures = texs, d.n_textures + 1
    out._keep = (nodes, mats, texs)
    return out


def _check_disjoint(gs, label):
    """1 spp: each pixel channel is non-zero in at most one group, and a NaN one is NaN in exactly one group."""
    nan = np.isnan(gs)
    live = nan | (gs != 0.0)
    assert (live.sum(axis=0) <= 1).all(), f"{label}: a pixel channel is non-zero in more than one group"
    assert (nan.sum(axis=0) <= 1).all(), label


CASES = [  # scene, width, flags
    ("cornel_box", 96, 0),                     # flat scan
    ("cornel_smoke", 96, 0),                   # flat scan + media
    ("simple_light", 128, 0),                  # flat scan, rich textures
    ("final_scene", 96, "lockstep"),           # lockstep tree, media, rich textures, a global fog sphere
    ("stress", 128, "persistent_wide"),        # 16 light nodes on the persistent kernel, 8-wide tree
    ("stress", 128, "persistent_binary"),      # ... and the binary tree
    ("enclosed", 64, 0),                       # the emitter is a global sky sphere under FlipFace
    ("enclosed", 64, "persistent_binary"),     # ... ended by k_wave_bvh's hit_globals
    ("lights", 96, 0),                         # an emissive AABox in a tree, a light under Translate / RotateY
    ("lights", 96, "no_tail"),
]


def _flags(api, f):
    return {"lockstep": api.FLAG_BVH_LOCKSTEP, "persistent_wide": api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_WIDE,
            "persistent_binary": api.FLAG_BVH_PERSISTENT | api.FLAG_BVH_BINARY, "no_tail": api.FLAG_NO_TAIL}.get(f, f)


@pytest.mark.parametrize("name,width,flags", CASES, ids=[f"{c[0]}-{c[2] or 'default'}" for c in CASES])
def test_groups_add_up_to_the_image(rt, gpu_ctx, name, width, flags):
    api = rt.api
    hs, cam, params = _scene(api, name)
    flags = _flags(api, flags)
    gsc = api.Scene(gpu_ctx, hs.desc)
    groups = api.light_groups_by_node(hs.desc)
    assert groups.n_groups >= 2
    if name == "stress":
        assert groups.n_groups == 17
    for s in range(8):
        p = params(width, s, s + 1, flags)
        gs, st = gsc.render_light_groups(cam, p, groups)
        assert gs.shape == (groups.n_groups, p.height, p.width, 3)
        _check_disjoint(gs, f"{name} sample {s}")
        check_identical_render((gs.sum(axis=0), None, st), gsc.render(cam, p), f"{name} sample {s}", 1, s)
    p = params(width, 0, 16, flags)
    gs, st = gsc.render_light_groups(cam, p, groups)
    check_identical_render((gs.sum(axis=0), None, st), gsc.render(cam, p), f"{name} 16 spp", 16)
    lit = [g for g in range(groups.n_groups) if np.nansum(gs[g]) > 0]
    print(f"[light groups {name}] {groups.n_groups} groups, {len(lit)} with light; {st.rays} rays")
    gsc.close()


SHARE_CASES = [  # scene, width, flags, what to double: a light node (by_node group) or a shared material (by_material group)
    ("cornel_box", 96, 0, "node"),
    ("stress", 128, "persistent_wide", "material"),
    ("enclosed", 64, 0, "node"),
    ("lights", 96, 0, "node"),
]


@pytest.mark.parametrize("name,width,flags,what", SHARE_CASES, ids=[f"{c[0]}-{c[3]}" for c in SHARE_CASES])
def test_each_group_is_its_lights_share(rt, gpu_ctx, name, width, flags, what):
    api = rt.api
    hs, cam, params = _scene(api, name)
    flags = _flags(api, flags)
    gsc = api.Scene(gpu_ctx, hs.desc)
    if what == "node":
        groups = api.light_groups_by_node(hs.desc)
        light = groups.members[0][0]
        relit = api.Scene(gpu_ctx, _relit_desc(api, hs.desc, node=light))
    else:
        groups = api.light_groups_by_material(hs.desc)
        assert groups.n_groups == 2 and len(groups.members[0]) == 16  # one material shared by the 16 lights
        d = hs.desc.contents
        relit = api.Scene(gpu_ctx, _relit_desc(api, hs.desc, material=d.nodes[groups.members[0][0]].material))
    scales = np.ones(groups.n_groups, np.float32)
    scales[0] = 2.0
    for s in range(4):
        p = params(width, s, s + 1, flags)
        gs, st = gsc.render_light_groups(cam, p, groups)
        check_identical_render((api.relight(gs, scales), None, st), relit.render(cam, p), f"{name}: group 0 doubled, sample {s}", 1, s)
    relit.close(), gsc.close()


def test_background_group_is_the_backgrounds_share(rt, gpu_ctx):
    api = rt.api
    hs, cam, params = _scene(api, "cornel_box")
    gsc = api.Scene(gpu_ctx, hs.desc)
    groups = api.light_groups_by_node(hs.desc)
    scales = np.ones(groups.n_groups, np.float32)
    scales[groups.background_group] = 2.0
    for s in range(4):
        p = params(96, s, s + 1)
        p.background[:] = [0.2, 0.3, 0.5]
        gs, st = gsc.render_light_groups(cam, p, groups)
        assert np.nansum(gs[groups.background_group]) > 0
        p2 = api.RenderParams.from_buffer_copy(p)
        p2.background[:] = [0.4, 0.6, 1.0]
        check_identical_render((api.relight(gs, scales), None, st), gsc.render(cam, p2), f"background doubled, sample {s}", 1, s)
    gsc.close()


def test_merged_groups_are_the_sums_of_their_parts(rt, gpu_ctx):
    """The two lights of the ad-hoc scene in one group, and per-RGB scales through relight."""
    api = rt.api
    hs, cam, params = _scene(api, "lights")
    gsc = api.Scene(gpu_ctx, hs.desc)
    sep = api.light_groups_by_node(hs.desc)
    assert sep.n_groups == 3
    merged = api.LightGroups(np.zeros_like(sep.table), 2, 1)  # both lights in group 0, the background in group 1
    for s in range(4):
        p = params(96, s, s + 1)
        a, sa = gsc.render_light_groups(cam, p, sep)
        b, sb = gsc.render_light_groups(cam, p, merged)
        assert sa.rays == sb.rays
        check_identical_sums(b, np.stack([a[0] + a[1], a[2]]), 1, f"merged lights, sample {s}", s)
    rgb = api.relight(a, [[1.0, 0.5, 0.25], [0.0, 0.0, 0.0], [1.0, 1.0, 1.0]])
    assert np.array_equal(rgb, (a[0] * np.float32([1.0, 0.5, 0.25]) + a[2]).astype(np.float32), equal_nan=True)
    gsc.close()


@pytest.mark.parametrize("name", ["cornel_box", "final_scene"])
def test_schedules_change_nothing(rt, gpu_ctx, name):
    """No tail kernel, pools of 2^16 and 4096 paths, sample ranges: the same paths, rays and sums (bit for bit at 1 spp)."""
    api = rt.api
    hs, cam, params = _scene(api, name)
    gsc = api.Scene(gpu_ctx, hs.desc)
    groups = api.light_groups_by_node(hs.desc)
    for s in (0, 5):
        ref = gsc.render_light_groups(cam, params(64, s, s + 1), groups)
        for label, p in (("no tail", params(64, s, s + 1, api.FLAG_NO_TAIL)), ("pool 2^16", params(64, s, s + 1, pool=1 << 16)),
                         ("pool 4096", params(64, s, s + 1, pool=4096))):
            gs, st = gsc.render_light_groups(cam, p, groups)
            check_identical_render((gs, None, st), (ref[0], None, ref[1]), f"{name} {label}, sample {s}", 1, s)
    lo, slo = gsc.render_light_groups(cam, params(64, 0, 4), groups)
    hi, shi = gsc.render_light_groups(cam, params(64, 4, 8), groups)
    whole, sall = gsc.render_light_groups(cam, params(64, 0, 8), groups)
    check_identical_sums(lo + hi, whole, 8, f"{name} [0,4) + [4,8)")
    assert slo.rays + shi.rays == sall.rays and slo.paths + shi.paths == sall.paths
    gsc.close()


def test_two_device_context(rt, gpu_ctx):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    api = rt.api
    hs, cam, params = _scene(api, "stress")
    groups = api.light_groups_by_node(hs.desc)
    one = api.Scene(gpu_ctx, hs.desc)
    ctx2 = api.Context([0, 1])
    two = api.Scene(ctx2, hs.desc)
    for s in (0, 1):
        p = params(96, s, s + 1)
        a, sa = one.render_light_groups(cam, p, groups)
        b, sb = two.render_light_groups(cam, p, groups)
        check_identical_render((b, None, sb), (a, None, sa), f"two devices, sample {s}", 1, s)
    p = params(96, 0, 8)
    a, sa = one.render_light_groups(cam, p, groups)
    b, sb = two.render_light_groups(cam, p, groups)
    check_identical_render((b, None, sb), (a, None, sa), "two devices, 8 spp", 8)
    two.close(), ctx2.close(), one.close()


def test_argument_checks(rt):
    import torch

    api = rt.api
    lib = api.load_library()
    ctx = api.Context(0)  # its own context: the 2^32-pixel call must not leave buffers behind
    hs = api.HostScene("cornel_box", seed=1)
    gsc = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    good = api.light_groups_by_node(hs.desc)
    light = good.members[0][0]
    out = np.zeros(good.n_groups * 16 * 16 * 3, np.float32)

    def status(groups=good, params=None, scene=gsc._h, camera=C.byref(cam), rgb=out.ctypes.data):
        params = hs.params(width=16, height=16, spp=2) if params is None else params
        return lib.rt1w_render_light_groups(scene, camera, C.byref(params) if params is not False else None,
                                            C.byref(groups) if groups is not None else None, rgb, None)

    def table(**kw):
        t = good.table.copy()
        for node, g in kw.get("entries", {}).items():
            t[node] = g
        return api.LightGroups(t, kw.get("n_groups", good.n_groups), kw.get("background", good.background_group))

    assert status() == api.OK
    assert status(table(entries={0: -7})) == api.OK  # entries of nodes that lower to no DiffuseLight primitive are not read
    assert status(scene=None) == api.ERR_INVALID
    assert status(camera=None) == api.ERR_INVALID
    assert status(params=False) == api.ERR_INVALID
    assert status(groups=None) == api.ERR_INVALID
    assert status(rgb=None) == api.ERR_INVALID
    short = api.LightGroups(good.table[:-1], good.n_groups, good.background_group)
    assert status(short) == api.ERR_INVALID  # n_nodes differs from the committed description's
    assert status(table(n_groups=0, background=0)) == api.ERR_INVALID
    assert status(table(background=-1)) == api.ERR_INVALID
    assert status(table(background=good.n_groups)) == api.ERR_INVALID
    assert status(table(entries={light: -1})) == api.ERR_INVALID
    assert status(table(entries={light: good.n_groups})) == api.ERR_INVALID
    reserved = table()
    reserved.reserved = 1
    assert status(reserved) == api.ERR_INVALID
    null_table = table()
    null_table.group_of_node = None
    assert status(null_table) == api.ERR_INVALID
    assert status(params=hs.params(width=16, height=16, spp=2, flags=api.FLAG_STATS)) == api.ERR_INVALID
    assert status(params=hs.params(width=0, height=16, spp=2)) == api.ERR_INVALID
    assert status(params=hs.params(width=16, height=16, sample_begin=4, sample_end=4)) == api.ERR_INVALID
    assert status(params=hs.params(width=16, height=16, spp=1 << 24)) == api.ERR_UNSUPPORTED
    # exactly 2^32 group pixels: refused before anything is allocated (its sums alone would take 48 GB)
    many = api.LightGroups(np.zeros(len(good.table), np.int32), 65536, 1)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(0)
    assert status(many, hs.params(width=256, height=256, spp=1), rgb=None) == api.ERR_INVALID
    free1, _ = torch.cuda.mem_get_info(0)
    assert free0 - free1 < (1 << 30), f"{(free0 - free1) / 2**30:.1f} GB allocated by a refused call"
    gsc.close(), ctx.close()


def test_demo_driver_writes_group_pfm_files(rt, gpu_ctx):
    """`rt1w_main cornel_box --spp 1 --light-groups PREFIX`: one PFM per group with the binding's group means bit for bit (at 1
    spp the sums do not depend on the order of the atomics), its groups on stderr, and the same P3 image as without it."""
    api = rt.api
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "rt1w_main")
    args = [exe, "cornel_box", "--width", "64", "--spp", "1"]
    plain = subprocess.run(args, capture_output=True, timeout=300)
    assert plain.returncode == 0, plain.stderr.decode()
    hs = api.HostScene("cornel_box", seed=1)
    groups = api.light_groups_by_node(hs.desc)
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "L")
        r = subprocess.run(args + ["--light-groups", prefix], capture_output=True, timeout=300)
        assert r.returncode == 0, r.stderr.decode()
        files = [api.read_pfm(f"{prefix}_group{k}.pfm") for k in range(groups.n_groups)]
        assert not os.path.exists(f"{prefix}_group{groups.n_groups}.pfm")
        for bad in (["--frames", "2"], ["--max-error", "1"], ["--denoise"]):
            assert subprocess.run(args + ["--light-groups", prefix] + bad, capture_output=True, timeout=60).returncode == 2
    assert r.stdout == plain.stdout
    err = r.stderr.decode()
    assert f"light group 0: node {groups.members[0][0]}" in err and f"light group {groups.n_groups - 1}: background" in err
    gsc = api.Scene(gpu_ctx, hs.desc)
    gs, _ = gsc.render_light_groups(hs.camera(), hs.params(width=64, spp=1, seed=0), groups)
    for k in range(groups.n_groups):
        want = np.where(np.isnan(gs[k]), np.float32(0), gs[k] / np.float32(1)).astype(np.float32)
        assert files[k].tobytes() == want.tobytes(), f"group {k}'s PFM differs from the binding's mean"
    gsc.close()
