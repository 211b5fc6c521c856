"""ctypes bindings of include/rt1w.h and host/host_api.h (see package docstring)."""
import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
BUILD_DIR = os.path.join(PKG_DIR, "_build")
LIB_PATH = os.environ.get("RT1W_LIB") or os.path.join(BUILD_DIR, "librt1w.so")  # RT1W_LIB: tuning variants only
HOST_LIB_PATH = os.path.join(BUILD_DIR, "librt1w_host.so")
ASSETS_DIR = os.path.join(os.path.dirname(PKG_DIR), "assets")

# --------------------------------------------------------------------------- enums
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NO_DEVICE, ERR_STATE = range(6)
(NODE_SPHERE, NODE_MOVING_SPHERE, NODE_XY_RECT, NODE_XZ_RECT, NODE_YZ_RECT, NODE_AABOX, NODE_TRANSLATE,
 NODE_ROTATE_Y, NODE_FLIP_FACE, NODE_CONSTANT_MEDIUM, NODE_BVH) = range(11)
MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_DIFFUSE_LIGHT, MAT_ISOTROPIC, MAT_NONE = range(6)
TEX_SOLID, TEX_CHECKER, TEX_NOISE, TEX_IMAGE, TEX_PERLIN = range(5)
FLAG_STATS = 1
FLAG_PROFILE = 2
FLAG_BVH_LOCKSTEP = 4
FLAG_BVH_PERSISTENT = 8
FLAG_BVH_BINARY = 16
FLAG_BVH_WIDE = 32
FLAG_NO_TAIL = 64

SCENE_IDS = {"random_scene": 0, "two_spheres": 1, "two_perlin_spheres": 2, "earth": 3, "simple_light": 4,
             "cornel_box": 5, "cornel_smoke": 6, "final_scene": 7, "stress": 8, "one_weekend": 9}


# --------------------------------------------------------------------------- structs (include/rt1w.h)
class Node(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("child_begin", C.c_int32), ("child_count", C.c_int32),
                ("p", C.c_double * 10)]


class Material(C.Structure):
    _fields_ = [("type", C.c_int32), ("texture", C.c_int32), ("albedo", C.c_double * 3), ("fuzz", C.c_double),
                ("ir", C.c_double)]


class Texture(C.Structure):
    _fields_ = [("type", C.c_int32), ("odd", C.c_int32), ("even", C.c_int32), ("table", C.c_int32),
                ("color", C.c_double * 3), ("scale", C.c_double)]


class Perlin(C.Structure):
    _fields_ = [("ranvec", (C.c_double * 3) * 256), ("perm_x", C.c_int32 * 256), ("perm_y", C.c_int32 * 256),
                ("perm_z", C.c_int32 * 256)]


class Image(C.Structure):
    _fields_ = [("rgb8", C.POINTER(C.c_uint8)), ("width", C.c_int32), ("height", C.c_int32)]


class SceneDesc(C.Structure):
    _fields_ = [("nodes", C.POINTER(Node)), ("n_nodes", C.c_int32),
                ("children", C.POINTER(C.c_int32)), ("n_children", C.c_int32),
                ("materials", C.POINTER(Material)), ("n_materials", C.c_int32),
                ("textures", C.POINTER(Texture)), ("n_textures", C.c_int32),
                ("perlins", C.POINTER(Perlin)), ("n_perlins", C.c_int32),
                ("images", C.POINTER(Image)), ("n_images", C.c_int32),
                ("world", C.c_int32), ("has_lights", C.c_int32),
                ("lights", C.POINTER(C.c_int32)), ("n_lights", C.c_int32)]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("lower_left_corner", C.c_double * 3), ("horizontal", C.c_double * 3),
                ("vertical", C.c_double * 3), ("u", C.c_double * 3), ("v", C.c_double * 3), ("w", C.c_double * 3),
                ("lens_radius", C.c_double), ("time0", C.c_double), ("time1", C.c_double)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("sample_begin", C.c_int32), ("sample_end", C.c_int32),
                ("max_depth", C.c_int32), ("flags", C.c_uint32), ("seed", C.c_uint64), ("background", C.c_double * 3),
                ("stat_clamp", C.c_double), ("pool_paths", C.c_int32), ("reserved", C.c_int32)]


KERNEL_NAMES = ["wave", "-", "-", "-", "-", "-", "-"]  # slot = 2 + rt1w_material_type for the shade kernels


class RenderStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("waves", C.c_uint64), ("launches", C.c_uint64),
                ("render_ms", C.c_double), ("kernel_ms", C.c_double * 7), ("kernel_launches", C.c_uint64 * 7)]


class SceneInfo(C.Structure):
    _fields_ = [("n_prims", C.c_int32), ("n_bvh_nodes", C.c_int32), ("n_frames", C.c_int32), ("n_lights", C.c_int32),
                ("bvh_depth", C.c_int32), ("material_mask", C.c_int32), ("build_ms", C.c_double),
                ("upload_ms", C.c_double), ("sah_cost", C.c_double), ("n_wide_nodes", C.c_int32), ("wide_depth", C.c_int32),
                ("wide_default", C.c_int32), ("n_global_prims", C.c_int32), ("wide_children", C.c_double)]


class FlatPrim(C.Structure):
    _fields_ = [("kind", C.c_int32), ("node", C.c_int32), ("material", C.c_int32), ("frame", C.c_int32),
                ("flags", C.c_int32), ("boundary", C.c_int32), ("p", C.c_double * 10),
                ("bbox_min", C.c_double * 3), ("bbox_max", C.c_double * 3), ("time0", C.c_double), ("time1", C.c_double)]


class Ray(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("direction", C.c_float * 3), ("time", C.c_float)]


RAY_DTYPE = np.dtype([("origin", np.float32, 3), ("direction", np.float32, 3), ("time", np.float32)])


class HostSettings(C.Structure):
    _fields_ = [("image_width", C.c_int32), ("image_height", C.c_int32), ("samples_per_pixel", C.c_int32),
                ("max_depth", C.c_int32), ("aspect_ratio", C.c_double), ("aperture", C.c_double),
                ("vfov_deg", C.c_double), ("background", C.c_double * 3), ("look_from", C.c_double * 3),
                ("look_at", C.c_double * 3)]


# every entry point include/rt1w.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "rt1w_abi_version", "rt1w_last_error", "rt1w_context_create", "rt1w_context_destroy", "rt1w_scene_create",
    "rt1w_scene_destroy", "rt1w_scene_get_info", "rt1w_scene_get_prims", "rt1w_scene_get_leaf_prims", "rt1w_lower_prims", "rt1w_lower_face_groups", "rt1w_render",
    "rt1w_render_device", "rt1w_render_rgb8", "rt1w_trace_closest", "rt1w_resolve_rgb8", "rt1w_philox4x32",
    "rt1w_context_create_multi", "rt1w_comm_unique_id", "rt1w_context_comm_init", "rt1w_context_get_comm", "rt1w_shard_sample_range",
    "rt1w_eval_light_pdf", "rt1w_eval_texture", "rt1w_eval_perlin", "rt1w_eval_dielectric", "rt1w_eval_scatter", "rt1w_build_bvh_host",
    "rt1w_render_adaptive", "rt1w_render_batch", "rt1w_render_aov", "rt1w_eval_camera_rays",
]


class Rt1wError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"rt1w status {status}: {message}")
        self.status = status


_lib = None
_host = None


def load_library():
    """Loads the product library.  No fallback: a missing build is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing — run `python raytracing-1w_b200/build.py` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.rt1w_abi_version.restype = C.c_int32
    lib.rt1w_last_error.restype = C.c_char_p
    lib.rt1w_context_create.argtypes = [C.c_int32, C.POINTER(vp)]
    lib.rt1w_context_destroy.argtypes = [vp]
    lib.rt1w_context_destroy.restype = None
    lib.rt1w_scene_create.argtypes = [vp, C.POINTER(SceneDesc), C.POINTER(vp)]
    lib.rt1w_scene_destroy.argtypes = [vp]
    lib.rt1w_scene_destroy.restype = None
    lib.rt1w_scene_get_info.argtypes = [vp, C.POINTER(SceneInfo)]
    lib.rt1w_scene_get_prims.argtypes = [vp, C.POINTER(FlatPrim), C.c_int32, C.POINTER(C.c_int32)]
    lib.rt1w_scene_get_leaf_prims.argtypes = [vp, vp, C.c_int32, C.POINTER(C.c_int32)]
    lib.rt1w_lower_prims.argtypes = [C.POINTER(SceneDesc), C.POINTER(FlatPrim), C.c_int32, C.POINTER(C.c_int32)]
    lib.rt1w_lower_face_groups.argtypes = [C.POINTER(SceneDesc), vp, vp, C.c_int32, C.POINTER(C.c_int32)]
    lib.rt1w_build_bvh_host.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, C.POINTER(C.c_int32), vp, vp, C.c_int32, C.POINTER(C.c_int32), vp,
                                        C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.rt1w_render.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, vp, C.POINTER(RenderStats)]
    lib.rt1w_render_device.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, vp, C.POINTER(RenderStats)]
    lib.rt1w_trace_closest.argtypes = [vp, vp, C.c_size_t, C.c_uint64, vp, vp, vp, vp, vp]
    lib.rt1w_render_rgb8.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, C.POINTER(RenderStats)]
    lib.rt1w_render_adaptive.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), C.c_int32, C.c_double, vp, vp, vp, vp,
                                         C.POINTER(RenderStats)]
    lib.rt1w_render_batch.argtypes = [vp, C.POINTER(Camera), C.c_int32, vp, C.POINTER(RenderParams), vp, vp, C.POINTER(RenderStats)]
    lib.rt1w_render_aov.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, vp, vp, vp, C.POINTER(RenderStats)]
    lib.rt1w_eval_camera_rays.argtypes = [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, vp, C.c_size_t, vp]
    lib.rt1w_resolve_rgb8.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.rt1w_resolve_rgb8.restype = None
    lib.rt1w_philox4x32.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.rt1w_philox4x32.restype = None
    lib.rt1w_context_create_multi.argtypes = [C.POINTER(C.c_int32), C.c_int32, C.POINTER(vp)]
    lib.rt1w_comm_unique_id.argtypes = [vp, C.c_size_t]
    lib.rt1w_context_comm_init.argtypes = [vp, vp, C.c_int32, C.c_int32]
    lib.rt1w_context_get_comm.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.rt1w_shard_sample_range.argtypes = [C.c_int32] * 4 + [C.POINTER(C.c_int32)] * 2
    lib.rt1w_shard_sample_range.restype = None
    lib.rt1w_eval_light_pdf.argtypes = [vp, C.c_int32, vp, vp, C.c_size_t, vp]
    lib.rt1w_eval_texture.argtypes = [vp, C.c_int32, vp, vp, C.c_size_t, vp]
    lib.rt1w_eval_perlin.argtypes = [vp, C.c_int32, C.c_int32, vp, C.c_size_t, vp]
    lib.rt1w_eval_dielectric.argtypes = [vp, vp, vp, vp, C.c_size_t, vp, vp, vp]
    lib.rt1w_eval_scatter.argtypes = [vp, vp, C.c_size_t, C.c_uint64, vp, vp, vp, vp, vp]
    _lib = lib
    return lib


def load_host_library():
    global _host
    if _host is not None:
        return _host
    if not os.path.exists(HOST_LIB_PATH):
        raise ImportError(f"{HOST_LIB_PATH} is missing — run `python raytracing-1w_b200/build.py`")
    h = C.CDLL(HOST_LIB_PATH)
    vp = C.c_void_p
    h.rt1w_host_scene_build.argtypes = [C.c_int32, C.c_uint64, vp, C.c_int32, C.c_int32, C.c_int32]
    h.rt1w_host_scene_build.restype = vp
    h.rt1w_host_scene_id.argtypes = [C.c_char_p]
    h.rt1w_host_scene_desc.argtypes = [vp]
    h.rt1w_host_scene_desc.restype = C.POINTER(SceneDesc)
    h.rt1w_host_scene_settings.argtypes = [vp, C.POINTER(HostSettings)]
    h.rt1w_host_scene_settings.restype = None
    h.rt1w_host_scene_camera.argtypes = [vp, C.c_double, C.POINTER(Camera)]
    h.rt1w_host_scene_camera.restype = None
    h.rt1w_host_scene_free.argtypes = [vp]
    h.rt1w_host_scene_free.restype = None
    h.rt1w_host_camera_new.argtypes = [C.POINTER(C.c_double)] * 3 + [C.c_double] * 6 + [C.POINTER(Camera)]
    h.rt1w_host_camera_new.restype = None
    h.rt1w_host_write_ppm.argtypes = [C.c_char_p, vp, C.c_int32, C.c_int32]
    h.rt1w_host_last_error.restype = C.c_char_p
    _host = h
    return h


def _check(status):
    if status != OK:
        raise Rt1wError(status, load_library().rt1w_last_error().decode())


def load_earthmap():
    """Decoded assets/earthmap (RGB8, row 0 = top) or None when the asset is absent."""
    path = os.path.join(ASSETS_DIR, "earthmap.ppm")
    if not os.path.exists(path):
        return None
    with open(path, "rb") as f:
        data = f.read()
    # P6 <w> <h> 255\n
    parts = data.split(b"\n", 3)
    assert parts[0] == b"P6"
    w, h = (int(x) for x in parts[1].split())
    px = np.frombuffer(parts[3], dtype=np.uint8, count=w * h * 3).reshape(h, w, 3).copy()
    return px


# --------------------------------------------------------------------------- host-side scene objects
class HostScene:
    """One arm of the reference's `match` (main.rs:815-937) built by the C++ mirror."""

    def __init__(self, name_or_id, seed=1, stress_spheres=0):
        h = load_host_library()
        which = SCENE_IDS[name_or_id] if isinstance(name_or_id, str) else int(name_or_id)
        earth = load_earthmap() if which in (3, 7) else None
        if which in (3, 7) and earth is None:
            raise FileNotFoundError("assets/earthmap.ppm missing (tools/prep_earthmap.py makes it)")
        self._earth = earth
        ptr = earth.ctypes.data_as(C.c_void_p) if earth is not None else None
        ew, eh = (earth.shape[1], earth.shape[0]) if earth is not None else (0, 0)
        self._h = h.rt1w_host_scene_build(which, seed, ptr, ew, eh, stress_spheres)
        if not self._h:
            raise RuntimeError("scene build failed: " + h.rt1w_host_last_error().decode())
        self.which = which
        self.settings = HostSettings()
        h.rt1w_host_scene_settings(self._h, C.byref(self.settings))

    @property
    def desc(self):
        return load_host_library().rt1w_host_scene_desc(self._h)

    def camera(self, aspect=None):
        cam = Camera()
        load_host_library().rt1w_host_scene_camera(self._h, self.settings.aspect_ratio if aspect is None else aspect,
                                                   C.byref(cam))
        return cam

    def params(self, width=None, height=None, spp=None, sample_begin=0, sample_end=None, seed=0, flags=0,
               stat_clamp=0.0, max_depth=None, pool_paths=0):
        s = self.settings
        p = RenderParams()
        p.width = s.image_width if width is None else width
        p.height = (int(p.width / s.aspect_ratio) if width is not None else s.image_height) if height is None else height
        spp = s.samples_per_pixel if spp is None else spp
        p.sample_begin = sample_begin
        p.sample_end = spp if sample_end is None else sample_end
        p.max_depth = s.max_depth if max_depth is None else max_depth
        p.flags = flags
        p.seed = seed
        p.background[:] = list(s.background)
        p.stat_clamp = stat_clamp
        p.pool_paths = pool_paths
        return p

    def close(self):
        if self._h:
            load_host_library().rt1w_host_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def camera_new(look_from, look_at, vup, vfov_deg, aspect, aperture, focus_dist, time0, time1):
    """Camera::new (camera.rs:22-59)."""
    cam = Camera()
    a3 = C.c_double * 3
    load_host_library().rt1w_host_camera_new(a3(*look_from), a3(*look_at), a3(*vup), vfov_deg, aspect, aperture,
                                             focus_dist, time0, time1, C.byref(cam))
    return cam


class DescBuilder:
    """Builds an rt1w_scene_desc from Python (tests use it for tiny ad-hoc scenes)."""

    def __init__(self):
        self.nodes, self.children, self.materials, self.textures, self.perlins, self.images = [], [], [], [], [], []
        self.lights, self.world, self.has_lights = [], -1, False
        self._keep = []

    # textures
    def solid(self, r, g, b):
        t = Texture(type=TEX_SOLID, odd=-1, even=-1, table=-1)
        t.color[:] = [r, g, b]
        self.textures.append(t)
        return len(self.textures) - 1

    def checker(self, odd, even):
        self.textures.append(Texture(type=TEX_CHECKER, odd=odd, even=even, table=-1))
        return len(self.textures) - 1

    def noise(self, scale, ranvec, perm_x, perm_y, perm_z, kind=TEX_NOISE):
        p = Perlin()
        for i in range(256):
            p.ranvec[i][:] = [float(x) for x in ranvec[i]]
        p.perm_x[:] = [int(x) for x in perm_x]
        p.perm_y[:] = [int(x) for x in perm_y]
        p.perm_z[:] = [int(x) for x in perm_z]
        self.perlins.append(p)
        self.textures.append(Texture(type=kind, odd=-1, even=-1, table=len(self.perlins) - 1, scale=scale))
        return len(self.textures) - 1

    def image(self, rgb8):
        arr = np.ascontiguousarray(rgb8, dtype=np.uint8)
        self._keep.append(arr)
        im = Image(rgb8=arr.ctypes.data_as(C.POINTER(C.c_uint8)), width=arr.shape[1], height=arr.shape[0])
        self.images.append(im)
        self.textures.append(Texture(type=TEX_IMAGE, odd=-1, even=-1, table=len(self.images) - 1))
        return len(self.textures) - 1

    # materials
    def _mat(self, type_, texture=-1, albedo=(0, 0, 0), fuzz=0.0, ir=0.0):
        m = Material(type=type_, texture=texture, fuzz=fuzz, ir=ir)
        m.albedo[:] = list(albedo)
        self.materials.append(m)
        return len(self.materials) - 1

    def lambertian(self, texture):
        return self._mat(MAT_LAMBERTIAN, texture)

    def metal(self, albedo, fuzz):
        return self._mat(MAT_METAL, albedo=albedo, fuzz=fuzz)

    def dielectric(self, ir):
        return self._mat(MAT_DIELECTRIC, ir=ir)

    def diffuse_light(self, texture):
        return self._mat(MAT_DIFFUSE_LIGHT, texture)

    def isotropic(self, texture):
        return self._mat(MAT_ISOTROPIC, texture)

    def null_material(self):
        return self._mat(MAT_NONE)

    # hittables
    def _node(self, type_, material, p, kids=()):
        n = Node(type=type_, material=material, child_begin=len(self.children), child_count=len(kids))
        for i, v in enumerate(p):
            n.p[i] = v
        self.children.extend(kids)
        self.nodes.append(n)
        return len(self.nodes) - 1

    def sphere(self, center, radius, material):
        return self._node(NODE_SPHERE, material, [*center, radius])

    def moving_sphere(self, c0, c1, t0, t1, radius, material):
        return self._node(NODE_MOVING_SPHERE, material, [*c0, *c1, t0, t1, radius])

    def xy_rect(self, x0, x1, y0, y1, k, material):
        return self._node(NODE_XY_RECT, material, [x0, x1, y0, y1, k])

    def xz_rect(self, x0, x1, z0, z1, k, material):
        return self._node(NODE_XZ_RECT, material, [x0, x1, z0, z1, k])

    def yz_rect(self, y0, y1, z0, z1, k, material):
        return self._node(NODE_YZ_RECT, material, [y0, y1, z0, z1, k])

    def aabox(self, p0, p1, material):
        return self._node(NODE_AABOX, material, [*p0, *p1])

    def translate(self, child, offset):
        return self._node(NODE_TRANSLATE, -1, list(offset), [child])

    def rotate_y(self, child, deg, time0=0.0, time1=1.0):
        return self._node(NODE_ROTATE_Y, -1, [deg, time0, time1], [child])

    def flip_face(self, child):
        return self._node(NODE_FLIP_FACE, -1, [], [child])

    def constant_medium(self, boundary, density, texture):
        return self._node(NODE_CONSTANT_MEDIUM, self.isotropic(texture), [density], [boundary])

    def bvh(self, kids, time0=0.0, time1=1.0):
        return self._node(NODE_BVH, -1, [time0, time1], list(kids))

    def set_world(self, node):
        self.world = node

    def set_lights(self, nodes):
        self.has_lights = True
        self.lights = list(nodes)

    def desc(self):
        d = SceneDesc()

        def arr(ctype, items):
            a = (ctype * max(1, len(items)))(*items)
            self._keep.append(a)
            return a

        d.nodes, d.n_nodes = arr(Node, self.nodes), len(self.nodes)
        d.children, d.n_children = arr(C.c_int32, self.children), len(self.children)
        d.materials, d.n_materials = arr(Material, self.materials), len(self.materials)
        d.textures, d.n_textures = arr(Texture, self.textures), len(self.textures)
        d.perlins, d.n_perlins = arr(Perlin, self.perlins), len(self.perlins)
        d.images, d.n_images = arr(Image, self.images), len(self.images)
        d.world = self.world
        d.has_lights = 1 if self.has_lights else 0
        d.lights, d.n_lights = arr(C.c_int32, self.lights), len(self.lights)
        self._keep.append(d)
        return d


def lower_prims(desc):
    """Host-side lowering (no GPU): the primitive table in primitive-id order."""
    lib = load_library()
    n = C.c_int32(0)
    dp = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
    _check(lib.rt1w_lower_prims(dp, None, 0, C.byref(n)))
    out = (FlatPrim * max(1, n.value))()
    _check(lib.rt1w_lower_prims(dp, out, n.value, C.byref(n)))
    return list(out)[: n.value]


# the binary tree's 32-byte node (csrc/bvh.h) and the 8-wide tree's 80-byte node (csrc/bvh8.h) as numpy records
BVH_NODE_DTYPE = np.dtype([("min", np.float32, 3), ("left_first", np.uint32), ("max", np.float32, 3), ("count", np.uint32)])
WIDE_NODE_DTYPE = np.dtype([("origin", np.float32, 3), ("exp", np.uint8, 3), ("imask", np.uint8), ("child_base", np.uint32),
                            ("prim_base", np.uint32), ("leaf_mask", np.uint32), ("unused", np.uint32), ("qlo", np.uint8, (3, 8)),
                            ("qhi", np.uint8, (3, 8))])


def build_bvh_host(bbox_min, bbox_max):
    """Host-side (no GPU): the SAH binary tree and its 8-wide collapse over n boxes, as scene commit builds them.
    -> dict(nodes, prim_order, wide_nodes, wide_leaf_remap, depth, wide_depth)."""
    lib = load_library()
    lo, hi = np.ascontiguousarray(bbox_min, dtype=np.float64), np.ascontiguousarray(bbox_max, dtype=np.float64)
    n = lo.shape[0]
    n_nodes, n_wide, depth, wide_depth = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    _check(lib.rt1w_build_bvh_host(lo.ctypes.data, hi.ctypes.data, n, None, 0, C.byref(n_nodes), None, None, 0, C.byref(n_wide), None,
                                   C.byref(depth), C.byref(wide_depth)))
    nodes, wide = np.zeros(n_nodes.value, dtype=BVH_NODE_DTYPE), np.zeros(n_wide.value, dtype=WIDE_NODE_DTYPE)
    order, remap = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
    _check(lib.rt1w_build_bvh_host(lo.ctypes.data, hi.ctypes.data, n, nodes.ctypes.data, n_nodes.value, C.byref(n_nodes), order.ctypes.data,
                                   wide.ctypes.data, n_wide.value, C.byref(n_wide), remap.ctypes.data, C.byref(depth), C.byref(wide_depth)))
    return dict(nodes=nodes, prim_order=order, wide_nodes=wide, wide_leaf_remap=remap, depth=depth.value, wide_depth=wide_depth.value)


def lower_face_groups(desc):
    """Host-side (no GPU): per lowered primitive the face group of the flat scan (-1: none) and its face; the group count."""
    lib = load_library()
    n_prims = len(lower_prims(desc))
    dp = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
    group, face = np.full(max(1, n_prims), -1, dtype=np.int32), np.full(max(1, n_prims), -1, dtype=np.int32)
    n_groups = C.c_int32(0)
    _check(lib.rt1w_lower_face_groups(dp, group.ctypes.data, face.ctypes.data, n_prims, C.byref(n_groups)))
    return group[:n_prims], face[:n_prims], n_groups.value


# --------------------------------------------------------------------------- device objects
COMM_ID_BYTES = 128


def comm_unique_id():
    """rt1w_comm_unique_id: the id rank 0 makes and the host side ships to the other ranks (one process per GPU)."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    _check(load_library().rt1w_comm_unique_id(buf, COMM_ID_BYTES))
    return bytes(buf)


def shard_sample_range(rank, n_ranks, sample_begin, sample_end):
    """rt1w_shard_sample_range: the library's split rule (host code)."""
    b, e = C.c_int32(), C.c_int32()
    load_library().rt1w_shard_sample_range(rank, n_ranks, sample_begin, sample_end, C.byref(b), C.byref(e))
    return b.value, e.value


class Context:
    """rt1w_context_create (one device) or, given a list of device ids, rt1w_context_create_multi (one process driving
    several GPUs: sample ranges sharded inside the library, NCCL reduce to the first device)."""

    def __init__(self, device_id=0):
        lib = load_library()
        self._h = C.c_void_p()
        if isinstance(device_id, (list, tuple)):
            ids = (C.c_int32 * len(device_id))(*device_id)
            _check(lib.rt1w_context_create_multi(ids, len(device_id), C.byref(self._h)))
        else:
            _check(lib.rt1w_context_create(device_id, C.byref(self._h)))

    def comm_init(self, unique_id, n_ranks, rank):
        """rt1w_context_comm_init: joins the communicator of a one-process-per-GPU job; render calls become collective."""
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        _check(load_library().rt1w_context_comm_init(self._h, buf, n_ranks, rank))

    def comm(self):
        """-> (rank, ranks, devices this context drives itself)."""
        r, n, d = C.c_int32(), C.c_int32(), C.c_int32()
        _check(load_library().rt1w_context_get_comm(self._h, C.byref(r), C.byref(n), C.byref(d)))
        return r.value, n.value, d.value

    def eval_dielectric(self, unit_dir, normal, ratio):
        """Device `reflect`, `refract`, `reflectance` (material.rs:94-96,114-125) for n unit directions / normals / index ratios."""
        uv, nn = np.ascontiguousarray(unit_dir, dtype=np.float32), np.ascontiguousarray(normal, dtype=np.float32)
        rr = np.ascontiguousarray(ratio, dtype=np.float32)
        n = rr.shape[0]
        refl, refr, f = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32)
        _check(load_library().rt1w_eval_dielectric(self._h, uv.ctypes.data, nn.ctypes.data, rr.ctypes.data, n, refl.ctypes.data, refr.ctypes.data,
                                                   f.ctypes.data))
        return refl, refr, f

    def close(self):
        if self._h:
            load_library().rt1w_context_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scene:
    """A committed device scene (rt1w_scene_create)."""

    def __init__(self, ctx, desc):
        lib = load_library()
        self._ctx = ctx
        self._h = C.c_void_p()
        dp = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
        _check(lib.rt1w_scene_create(ctx._h, dp, C.byref(self._h)))

    def info(self):
        i = SceneInfo()
        _check(load_library().rt1w_scene_get_info(self._h, C.byref(i)))
        return i

    def prims(self):
        lib = load_library()
        n = C.c_int32(0)
        _check(lib.rt1w_scene_get_prims(self._h, None, 0, C.byref(n)))
        out = (FlatPrim * max(1, n.value))()
        _check(lib.rt1w_scene_get_prims(self._h, out, n.value, C.byref(n)))
        return list(out)[: n.value]

    def leaf_prims(self):
        """rt1w_scene_get_leaf_prims: the primitive id of every device leaf (the render keys media draws on the leaf index)."""
        lib = load_library()
        n = C.c_int32(0)
        _check(lib.rt1w_scene_get_leaf_prims(self._h, None, 0, C.byref(n)))
        out = np.empty(max(1, n.value), np.int32)
        _check(lib.rt1w_scene_get_leaf_prims(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out[: n.value]

    def render(self, camera, params, want_stat=False):
        """rt1w_render with HOST buffers; returns (rgb_sum[h,w,3] float32, stat or None, RenderStats)."""
        lib = load_library()
        out = np.empty((params.height, params.width, 3), dtype=np.float32)
        stat = np.empty((params.height, params.width, 6), dtype=np.float32) if want_stat else None
        st = RenderStats()
        _check(lib.rt1w_render(self._h, C.byref(camera), C.byref(params), out.ctypes.data_as(C.c_void_p),
                               stat.ctypes.data_as(C.c_void_p) if want_stat else None, C.byref(st)))
        return out, stat, st

    def render_into(self, camera, params, out, stat=None):
        """rt1w_render into caller-provided (e.g. pinned) host arrays."""
        st = RenderStats()
        _check(load_library().rt1w_render(self._h, C.byref(camera), C.byref(params), C.c_void_p(out.ctypes.data) if out is not None else None,
                                          C.c_void_p(stat.ctypes.data) if stat is not None else None, C.byref(st)))
        return st

    def render_rgb8(self, camera, params):
        """rt1w_render_rgb8: render + resolve on the device; returns (rgb8[h,w,3] uint8, RenderStats)."""
        out = np.empty((params.height, params.width, 3), dtype=np.uint8)
        st = RenderStats()
        _check(load_library().rt1w_render_rgb8(self._h, C.byref(camera), C.byref(params), out.ctypes.data_as(C.c_void_p), C.byref(st)))
        return out, st

    def render_adaptive(self, camera, params, min_spp, max_error, want_stat=False):
        """rt1w_render_adaptive: each pixel rendered until its 8-bit value has converged (params.sample_end = the cap).
        Returns (rgb_sum[h,w,3] float32, spp[h,w] int32, rgb8[h,w,3] uint8, stat[h,w,6] or None, RenderStats)."""
        h, w = params.height, params.width
        out, spp, rgb8 = np.empty((h, w, 3), np.float32), np.empty((h, w), np.int32), np.empty((h, w, 3), np.uint8)
        stat = np.empty((h, w, 6), np.float32) if want_stat else None
        st = RenderStats()
        _check(load_library().rt1w_render_adaptive(self._h, C.byref(camera), C.byref(params), min_spp, max_error, out.ctypes.data, spp.ctypes.data,
                                                   rgb8.ctypes.data, stat.ctypes.data if want_stat else None, C.byref(st)))
        return out, spp, rgb8, stat, st

    def render_batch(self, cameras, params, seeds=None):
        """rt1w_render_batch: one frame per camera, all in one wavefront; frame f uses seeds[f] (every frame params.seed when
        seeds is None).  Returns (rgb_sum[n,h,w,3] float32, rgb8[n,h,w,3] uint8, RenderStats)."""
        n, h, w = len(cameras), params.height, params.width
        cams = (Camera * max(n, 1))(*cameras)
        seed_arr = None if seeds is None else np.ascontiguousarray(seeds, dtype=np.uint64)
        if seed_arr is not None and seed_arr.shape != (n,):
            raise ValueError("seeds must hold one seed per camera")
        out, rgb8 = np.empty((n, h, w, 3), np.float32), np.empty((n, h, w, 3), np.uint8)
        st = RenderStats()
        _check(load_library().rt1w_render_batch(self._h, cams, n, seed_arr.ctypes.data if seed_arr is not None else None, C.byref(params),
                                                out.ctypes.data, rgb8.ctypes.data, C.byref(st)))
        return out, rgb8, st

    def render_aov(self, camera, params):
        """rt1w_render_aov: first-hit feature buffers, summed over the sample range.  Returns (albedo_sum[h,w,3],
        normal_sum[h,w,3], distance_sum[h,w], hits[h,w]) float32 and RenderStats; aov_means turns them into means."""
        h, w = params.height, params.width
        albedo, normal = np.empty((h, w, 3), np.float32), np.empty((h, w, 3), np.float32)
        distance, hits = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
        st = RenderStats()
        _check(load_library().rt1w_render_aov(self._h, C.byref(camera), C.byref(params), albedo.ctypes.data, normal.ctypes.data, distance.ctypes.data,
                                              hits.ctypes.data, C.byref(st)))
        return albedo, normal, distance, hits, st

    def eval_camera_rays(self, camera, params, pixel_seed, sample):
        """rt1w_eval_camera_rays: the render's first ray of path (pixel seed j*w+i, global sample index) -> RAY_DTYPE array."""
        seeds, samples = np.ascontiguousarray(pixel_seed, dtype=np.uint32), np.ascontiguousarray(sample, dtype=np.int32)
        if seeds.shape != samples.shape or seeds.ndim != 1:
            raise ValueError("pixel_seed and sample must be 1-d arrays of one length")
        out = np.empty(seeds.shape[0], dtype=RAY_DTYPE)
        _check(load_library().rt1w_eval_camera_rays(self._h, C.byref(camera), C.byref(params), seeds.ctypes.data, samples.ctypes.data, seeds.shape[0],
                                                    out.ctypes.data))
        return out

    def render_device(self, camera, params, d_ptr, stream=0):
        st = RenderStats()
        _check(load_library().rt1w_render_device(self._h, C.byref(camera), C.byref(params), C.c_void_p(d_ptr),
                                                 C.c_void_p(stream), C.byref(st)))
        return st

    def trace_closest(self, rays, seed=0):
        lib = load_library()
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        n = rays.shape[0]
        prim = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        normal = np.empty((n, 3), dtype=np.float32)
        ff = np.empty(n, dtype=np.uint8)
        uv = np.empty((n, 2), dtype=np.float32)
        _check(lib.rt1w_trace_closest(self._h, rays.ctypes.data_as(C.c_void_p), n, seed,
                                      prim.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p),
                                      normal.ctypes.data_as(C.c_void_p), ff.ctypes.data_as(C.c_void_p),
                                      uv.ctypes.data_as(C.c_void_p)))
        return prim, t, normal, ff, uv

    # pointwise parity hooks (include/rt1w.h: rt1w_eval_*)
    def eval_light_pdf(self, origins, dirs, light=-1):
        o, v = np.ascontiguousarray(origins, dtype=np.float64), np.ascontiguousarray(dirs, dtype=np.float32)
        n = o.shape[0]
        out = np.empty(n, np.float32)
        _check(load_library().rt1w_eval_light_pdf(self._h, light, o.ctypes.data, v.ctypes.data, n, out.ctypes.data))
        return out

    def eval_texture(self, texture, points, uv=None):
        p = np.ascontiguousarray(points, dtype=np.float64)
        n = p.shape[0]
        uv = None if uv is None else np.ascontiguousarray(uv, dtype=np.float32)
        out = np.empty((n, 3), np.float32)
        _check(load_library().rt1w_eval_texture(self._h, texture, p.ctypes.data, None if uv is None else uv.ctypes.data, n, out.ctypes.data))
        return out

    def eval_perlin(self, table, points, turb_depth=0):
        p = np.ascontiguousarray(points, dtype=np.float64)
        out = np.empty(p.shape[0], np.float32)
        _check(load_library().rt1w_eval_perlin(self._h, table, turb_depth, p.ctypes.data, p.shape[0], out.ctypes.data))
        return out

    def eval_scatter(self, rays, seed=0):
        """-> prim_id, material_type, scattered direction, weight (or emitted radiance), scattered time."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        n = rays.shape[0]
        prim, mat = np.empty(n, np.int32), np.empty(n, np.int32)
        d, w, t = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32)
        _check(load_library().rt1w_eval_scatter(self._h, rays.ctypes.data, n, seed, prim.ctypes.data, mat.ctypes.data, d.ctypes.data,
                                                w.ctypes.data, t.ctypes.data))
        return prim, mat, d, w, t

    def close(self):
        if self._h:
            load_library().rt1w_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def philox4x32(counter, key):
    """One Philox4x32-10 block (rt1w_philox4x32): what the device draws for (counter, key)."""
    c, k, o = (C.c_uint32 * 4)(*[int(x) & 0xFFFFFFFF for x in counter]), (C.c_uint32 * 2)(*[int(x) & 0xFFFFFFFF for x in key]), (C.c_uint32 * 4)()
    load_library().rt1w_philox4x32(c, k, o)
    return list(o)


def resolve_rgb8(rgb_sum, spp):
    """Color::into_sampled + Display for SampledColor (color.rs:14-21,56-65)."""
    lib = load_library()
    rgb_sum = np.ascontiguousarray(rgb_sum, dtype=np.float32)
    h, w, _ = rgb_sum.shape
    out = np.empty((h, w, 3), dtype=np.uint8)
    lib.rt1w_resolve_rgb8(rgb_sum.ctypes.data_as(C.c_void_p), w, h, spp, out.ctypes.data_as(C.c_void_p))
    return out


def aov_means(albedo_sum, normal_sum, distance_sum, hits, n_samples):
    """Means of rt1w_render_aov's sums over n_samples samples: albedo and normal / n (the normal is not renormalised),
    distance / hits (0 where no sample hit).  -> (albedo, normal, distance) float32."""
    n = np.float32(n_samples)
    hits = np.asarray(hits, dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        distance = np.where(hits > 0, np.asarray(distance_sum, dtype=np.float32) / np.where(hits > 0, hits, np.float32(1)), np.float32(0))
    return np.asarray(albedo_sum, np.float32) / n, np.asarray(normal_sum, np.float32) / n, distance.astype(np.float32)


def write_pfm(path, array):
    """Little-endian PFM (the HDR format common denoisers read): (h,w,3) -> "PF", (h,w) -> "Pf"; row 0 of the array is the
    top of the image (PFM stores the bottom row first)."""
    a = np.asarray(array, dtype=np.float32)
    if a.ndim == 3 and a.shape[2] == 3:
        kind = b"PF"
    elif a.ndim == 2:
        kind = b"Pf"
    else:
        raise ValueError("write_pfm takes an (h, w, 3) or (h, w) array")
    with open(path, "wb") as f:
        f.write(kind + b"\n%d %d\n-1.0\n" % (a.shape[1], a.shape[0]))
        f.write(np.ascontiguousarray(a[::-1]).astype("<f4").tobytes())


def read_pfm(path):
    """A PFM file (either byte order) as float32, row 0 = top: (h,w,3) for "PF", (h,w) for "Pf"."""
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = (int(x) for x in f.readline().split())
        scale = float(f.readline())
        data = np.frombuffer(f.read(), dtype="<f4" if scale < 0 else ">f4")
    shape = (h, w, 3) if kind == b"PF" else (h, w)
    return data[: int(np.prod(shape))].reshape(shape)[::-1].astype(np.float32)


def write_ppm(path, rgb8):
    h, w, _ = rgb8.shape
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    rc = load_host_library().rt1w_host_write_ppm(path.encode(), rgb8.ctypes.data_as(C.c_void_p), w, h)
    if rc != 0:
        raise IOError(load_host_library().rt1w_host_last_error().decode())
