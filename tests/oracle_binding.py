"""ctypes binding of the CPU oracle (oracle/_build/liboracle.so).

TEST INFRASTRUCTURE: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module.  The product never does.
"""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "_build", "liboracle.so")

rt = importlib.import_module("raytracing-1w_b200")
api = rt.api


class OracleStats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("seconds", C.c_double), ("threads", C.c_int32),
                ("reserved", C.c_int32)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(ORACLE_LIB):
        subprocess.check_call(["make", "-C", ORACLE_DIR])
    lib = C.CDLL(ORACLE_LIB)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.oracle_last_error.restype = C.c_char_p
    lib.oracle_scene_load.argtypes = [C.POINTER(api.SceneDesc), C.c_uint64]
    lib.oracle_scene_load.restype = vp
    lib.oracle_scene_free.argtypes = [vp]
    lib.oracle_scene_free.restype = None
    lib.oracle_scene_num_prims.argtypes = [vp]
    lib.oracle_scene_bvh_shape.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.oracle_scene_bvh_shape.restype = None
    lib.oracle_trace_closest.argtypes = [vp, vp, C.c_size_t, C.c_uint64, vp, vp, vp, vp, vp, vp, C.c_int32]
    lib.oracle_render.argtypes = [vp, C.POINTER(api.Camera), C.POINTER(api.RenderParams), C.c_int32, vp, vp,
                                  C.POINTER(OracleStats)]
    lib.oracle_replay_paths.argtypes = [vp, C.POINTER(api.Camera), C.POINTER(api.RenderParams), vp, C.c_size_t, vp, vp, C.c_int32,
                                        C.c_int32, vp, vp, vp]
    lib.oracle_replay_path_log.argtypes = [vp, C.POINTER(api.Camera), C.POINTER(api.RenderParams), vp, C.c_uint32, C.c_int32, C.c_int32,
                                           C.c_char_p, C.c_size_t]
    lib.oracle_replay_camera_rays.argtypes = [vp, C.POINTER(api.Camera), C.POINTER(api.RenderParams), C.c_size_t, vp, vp, C.c_int32, vp, vp,
                                              vp]
    lib.oracle_replay_camera_rays.restype = None
    lib.oracle_xz_rect_pdf_value.argtypes = [dp, dp, dp]
    lib.oracle_xz_rect_pdf_value.restype = C.c_double
    lib.oracle_sphere_pdf_value.argtypes = [dp, C.c_double, dp, dp]
    lib.oracle_sphere_pdf_value.restype = C.c_double
    lib.oracle_sphere_hit_t.argtypes = [dp, C.c_double, dp, dp, C.c_double, C.c_double]
    lib.oracle_sphere_hit_t.restype = C.c_double
    lib.oracle_reflectance.argtypes = [C.c_double, C.c_double]
    lib.oracle_reflectance.restype = C.c_double
    lib.oracle_refract.argtypes = [dp, dp, C.c_double, dp]
    lib.oracle_refract.restype = None
    lib.oracle_sphere_uv.argtypes = [dp, dp]
    lib.oracle_sphere_uv.restype = None
    lib.oracle_onb_from_w.argtypes = [dp, dp]
    lib.oracle_onb_from_w.restype = None
    lib.oracle_quantise.argtypes = [dp, C.c_int32, C.POINTER(C.c_int32)]
    lib.oracle_quantise.restype = None
    lib.oracle_camera_ray.argtypes = [C.POINTER(api.Camera), C.c_double, C.c_double, dp, dp]
    lib.oracle_camera_ray.restype = None
    lib.oracle_rotate_y_bbox.argtypes = [dp, dp, C.c_double, dp, dp]
    lib.oracle_rotate_y_bbox.restype = None
    lib.oracle_hit_one.argtypes = [vp, dp, dp, C.c_double, dp, dp, dp, C.POINTER(C.c_int32)]
    lib.oracle_perlin_noise.argtypes = [C.POINTER(api.Perlin), dp]
    lib.oracle_perlin_noise.restype = C.c_double
    lib.oracle_perlin_turb.argtypes = [C.POINTER(api.Perlin), dp, C.c_int32]
    lib.oracle_perlin_turb.restype = C.c_double
    lib.oracle_texture_value.argtypes = [vp, C.c_int32, C.c_double, C.c_double, dp, dp]
    lib.oracle_texture_value.restype = None
    lib.oracle_bvh_count.argtypes = [C.c_int32, C.c_uint64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.oracle_bvh_count.restype = None
    lib.oracle_chacha_block.argtypes = [vp, C.c_int32, vp]
    lib.oracle_chacha_block.restype = None
    lib.oracle_stdrng_u32.argtypes = [C.c_uint64, C.c_int32, vp]
    lib.oracle_stdrng_u32.restype = None
    lib.oracle_stdrng_from_seed_u32.argtypes = [vp, C.c_int32, vp]
    lib.oracle_stdrng_from_seed_u32.restype = None
    lib.oracle_stdrng_f64.argtypes = [C.c_uint64, C.c_int32, vp]
    lib.oracle_stdrng_f64.restype = None
    lib.oracle_philox.argtypes = [vp, vp, vp]
    lib.oracle_philox.restype = None
    _lib = lib
    return lib


def d3(*v):
    return (C.c_double * len(v))(*v)


class OracleScene:
    def __init__(self, desc, bvh_seed=7):
        lib = load()
        dp = desc if isinstance(desc, C.POINTER(api.SceneDesc)) else C.pointer(desc)
        self._h = lib.oracle_scene_load(dp, bvh_seed)
        if not self._h:
            raise RuntimeError("oracle_scene_load: " + lib.oracle_last_error().decode())

    @property
    def num_prims(self):
        return load().oracle_scene_num_prims(self._h)

    def bvh_shape(self):
        n, d = C.c_int32(), C.c_int32()
        load().oracle_scene_bvh_shape(self._h, C.byref(n), C.byref(d))
        return n.value, d.value

    def trace_closest(self, rays, seed=0, threads=0):
        rays = np.ascontiguousarray(rays, dtype=api.RAY_DTYPE)
        n = rays.shape[0]
        prim = np.empty(n, np.int32)
        t = np.empty(n, np.float64)
        normal = np.empty((n, 3), np.float64)
        ff = np.empty(n, np.uint8)
        uv = np.empty((n, 2), np.float64)
        amb = np.empty(n, np.uint8)
        rc = load().oracle_trace_closest(self._h, rays.ctypes.data, n, seed, prim.ctypes.data, t.ctypes.data,
                                         normal.ctypes.data, ff.ctypes.data, uv.ctypes.data, amb.ctypes.data, threads)
        assert rc == 0
        return prim, t, normal, ff, uv, amb

    def render(self, camera, params, threads=0, want_stat=False):
        out = np.empty((params.height, params.width, 3), np.float64)
        stat = np.empty((params.height, params.width, 6), np.float64) if want_stat else None
        st = OracleStats()
        rc = load().oracle_render(self._h, C.byref(camera), C.byref(params), threads, out.ctypes.data,
                                  stat.ctypes.data if want_stat else None, C.byref(st))
        assert rc == 0
        return out, stat, st

    def replay_paths(self, camera, params, pixel_seed, sample, leaf_of_prim=None, mutation=0, threads=0):
        """oracle_replay_paths: the render's paths (pixel seed j*w+i, global sample index) with the product's Philox draws.
        leaf_of_prim: device leaf index per primitive id (replay_leaf_map).  Returns (rgb[n,3] f64, rays[n] u32, flags[n] u8)."""
        seeds, samples = np.ascontiguousarray(pixel_seed, np.uint32), np.ascontiguousarray(sample, np.int32)
        assert seeds.shape == samples.shape and seeds.ndim == 1
        n = seeds.shape[0]
        lmap = None if leaf_of_prim is None else np.ascontiguousarray(leaf_of_prim, np.int32)
        rgb, rays, flags = np.empty((n, 3), np.float64), np.empty(n, np.uint32), np.empty(n, np.uint8)
        rc = load().oracle_replay_paths(self._h, C.byref(camera), C.byref(params), None if lmap is None else lmap.ctypes.data, n,
                                        seeds.ctypes.data, samples.ctypes.data, mutation, threads, rgb.ctypes.data, rays.ctypes.data,
                                        flags.ctypes.data)
        assert rc == 0, "oracle_replay_paths: " + load().oracle_last_error().decode()
        return rgb, rays, flags

    def replay_path_log(self, camera, params, pixel_seed, sample, leaf_of_prim=None, mutation=0):
        """One replayed path, bounce by bounce, as text."""
        lmap = None if leaf_of_prim is None else np.ascontiguousarray(leaf_of_prim, np.int32)
        buf = C.create_string_buffer(1 << 16)
        rc = load().oracle_replay_path_log(self._h, C.byref(camera), C.byref(params), None if lmap is None else lmap.ctypes.data,
                                           int(pixel_seed), int(sample), mutation, buf, len(buf))
        assert rc == 0, "oracle_replay_path_log: " + load().oracle_last_error().decode()
        return buf.value.decode()

    def replay_camera_rays(self, camera, params, pixel_seed, sample, mutation=0):
        """The replay's camera rays: (origin[n,3], direction[n,3], time[n]) f64."""
        seeds, samples = np.ascontiguousarray(pixel_seed, np.uint32), np.ascontiguousarray(sample, np.int32)
        n = seeds.shape[0]
        o, d, t = np.empty((n, 3)), np.empty((n, 3)), np.empty(n)
        load().oracle_replay_camera_rays(self._h, C.byref(camera), C.byref(params), n, seeds.ctypes.data, samples.ctypes.data, mutation,
                                         o.ctypes.data, d.ctypes.data, t.ctypes.data)
        return o, d, t

    def hit_one(self, o, d, time=0.0):
        t = C.c_double()
        p, n = d3(0, 0, 0), d3(0, 0, 0)
        ff = C.c_int32()
        prim = load().oracle_hit_one(self._h, d3(*o), d3(*d), time, C.byref(t), p, n, C.byref(ff))
        return prim, t.value, list(p), list(n), bool(ff.value)

    def texture_value(self, texture, u, v, p):
        out = d3(0, 0, 0)
        load().oracle_texture_value(self._h, texture, u, v, d3(*p), out)
        return list(out)

    def close(self):
        if self._h:
            load().oracle_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def replay_leaf_map(leaf_prims, n_prims):
    """Inverts rt1w_scene_get_leaf_prims (primitive id of each device leaf) into the leaf index of each primitive id, the
    table oracle_replay_paths keys media draws with.  Primitives without a leaf of their own (box sides after the first) get -1."""
    out = np.full(max(n_prims, 1), -1, np.int32)
    lp = np.asarray(leaf_prims, np.int64)
    ok = (lp >= 0) & (lp < n_prims)
    out[lp[ok]] = np.flatnonzero(ok).astype(np.int32)
    return out
