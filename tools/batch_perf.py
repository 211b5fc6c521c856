"""What one batch render (rt1w_render_batch) gains over a loop of rt1w_render calls on the same cameras and seeds.

    python tools/batch_perf.py [--repeats R] [--out FILE]

Cases:
  C1      Cornell box 600x600 x 16 spp, 32 frames of one camera with 32 seeds (the same work either way)
  turn    random_scene 1200x800 x 8 spp, a 16-frame turntable (look_from turned about the vertical axis through look_at)
  views   final_scene 256x256 x 32 spp, 64 views (a 64-frame turntable)
Per case and mode: wall-clock ms of the whole call sequence (each call ends with its sums on the host), median of R after
one warm-up; Mpaths/s; waves and launches summed over the calls; and whether the two give the same sums (NaNs in the same
places, the rest within 1e-4: the order of the fp32 additions differs).  Prints one JSON line per case; the GPU's name and
power limit are read (a query only) and printed with them.
"""
import argparse
import ctypes as C
import importlib
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [("C1", "cornel_box", 600, 600, 16, 32, "seeds"), ("turn", "random_scene", 1200, 800, 8, 16, "turntable"),
         ("views", "final_scene", 256, 256, 32, 64, "turntable")]


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True, timeout=30)
        return out.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def turntable(api, hs, n):
    s = hs.settings
    lf, la = np.array(s.look_from[:]), np.array(s.look_at[:])
    arm, cams = lf - la, []
    for k in range(n):
        a = 2.0 * math.pi * k / n
        eye = la + np.array([math.cos(a) * arm[0] + math.sin(a) * arm[2], arm[1], -math.sin(a) * arm[0] + math.cos(a) * arm[2]])
        cams.append(api.camera_new(eye.tolist(), la.tolist(), [0.0, 1.0, 0.0], s.vfov_deg, s.aspect_ratio, s.aperture, 10.0, 0.0, 1.0))
    return cams


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    api = importlib.import_module("raytracing-1w_b200").api
    lib = api.load_library()
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    ctx = api.Context(0)
    lines = []
    for name, scene_name, w, h, spp, n, kind in CASES:
        hs = api.HostScene(scene_name, seed=1)
        sc = api.Scene(ctx, hs.desc)
        cams = [hs.camera()] * n if kind == "seeds" else turntable(api, hs, n)
        seeds = np.arange(1, n + 1, dtype=np.uint64)
        p = hs.params(width=w, height=h, spp=spp)
        loop_out, batch_out = np.empty((n, h, w, 3), np.float32), np.empty((n, h, w, 3), np.float32)
        cam_arr = (api.Camera * n)(*cams)

        def loop():
            st_all = []
            for f in range(n):
                q = api.RenderParams.from_buffer_copy(p)
                q.seed = int(seeds[f])
                st_all.append(sc.render_into(cams[f], q, loop_out[f]))
            return st_all

        def batch():
            st = api.RenderStats()
            api._check(lib.rt1w_render_batch(sc._h, cam_arr, n, seeds.ctypes.data, C.byref(p), batch_out.ctypes.data, None, C.byref(st)))
            return [st]

        def timed(fn):
            fn()  # warm-up
            ms, stats = [], None
            for _ in range(args.repeats):
                t0 = time.perf_counter()
                stats = fn()
                ms.append(1e3 * (time.perf_counter() - t0))
            return float(np.median(ms)), stats

        rec = {"case": name, "scene": scene_name, "width": w, "height": h, "spp": spp, "frames": n, "cameras": kind}
        paths = n * w * h * spp
        for mode, fn in (("loop", loop), ("batch", batch)):
            ms, stats = timed(fn)
            rec[mode] = {"ms": round(ms, 2), "mpaths_s": round(paths / ms / 1e3, 1), "waves": int(sum(s.waves for s in stats)),
                         "launches": int(sum(s.launches for s in stats)), "rays": int(sum(s.rays for s in stats)),
                         "render_ms": round(sum(s.render_ms for s in stats), 2)}
        rec["speedup"] = round(rec["loop"]["ms"] / rec["batch"]["ms"], 3)
        nan_same = bool((np.isnan(loop_out) == np.isnan(batch_out)).all())
        ok = ~np.isnan(loop_out)
        rec["same_sums"] = nan_same and bool(np.allclose(loop_out[ok], batch_out[ok], rtol=1e-4, atol=1e-4))
        rec["same_rays"] = rec["loop"]["rays"] == rec["batch"]["rays"]
        rec["gpu"] = info
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        sc.close()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
