"""What the first-hit feature buffers (rt1w_render_aov) cost next to the render of the same camera, size and sample count.

    python tools/aov_perf.py [--repeats R] [--out FILE]

Cases: the six scenes of DESIGN.md section 13's A/B table at its sizes and sample counts, then a small image at a high sample
count (Cornell box 256^2 x 1024 spp: several lanes share a pixel) and a 4K image at one sample (a pixel per lane).
Per case: the device-resident render (rt1w_render_device) and the AOV call, each warmed up once and then timed R times;
the median of the device time between the call's CUDA events (render_ms: the AOV call's host copies are outside it) and
of the wall-clock ms of the whole call; rays and Grays/s (closest-hit queries per second: one per sample for the AOV call);
and aov / render, the ratio of the two device times.  Prints one JSON line per case; the GPU's name, power limit and max SM
clock are read (a query only) in the same run and printed first and with every line.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [  # name, scene, constructor arguments, width, height, spp
    ("C1", "cornel_box", {}, 600, 600, 100), ("random_scene", "random_scene", {}, 1200, 800, 8),
    ("one_weekend", "one_weekend", {}, 1200, 800, 32), ("final_scene", "final_scene", {}, 800, 800, 16),
    ("cornel_smoke", "cornel_smoke", {}, 600, 600, 32), ("stress", "stress", dict(stress_spheres=1_000_000), 1920, 1080, 8),
    ("small_high_spp", "cornel_box", {}, 256, 256, 1024), ("4k_1spp", "cornel_box", {}, 3840, 2160, 1),
]


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True, timeout=30)
        return out.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    api = importlib.import_module("raytracing-1w_b200").api
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    ctx = api.Context(0)
    lines = []
    for name, scene_name, kw, w, h, spp in CASES:
        hs = api.HostScene(scene_name, seed=1, **kw)
        sc = api.Scene(ctx, hs.desc)
        cam = hs.camera()
        p = hs.params(width=w, height=h, spp=spp, seed=1)
        d_sum = torch.empty(h * w * 3, dtype=torch.float32, device="cuda:0")

        def timed(fn):
            fn()  # warm-up
            dev, wall, st = [], [], None
            for _ in range(args.repeats):
                t0 = time.perf_counter()
                st = fn()
                wall.append(1e3 * (time.perf_counter() - t0))
                dev.append(st.render_ms)
            return float(np.median(dev)), float(np.median(wall)), st

        rec = {"case": name, "scene": scene_name, "width": w, "height": h, "spp": spp}
        for mode, fn in (("render", lambda: sc.render_device(cam, p, d_sum.data_ptr())), ("aov", lambda: sc.render_aov(cam, p)[4])):
            ms, wall_ms, st = timed(fn)
            rec[mode] = {"ms": round(ms, 3), "wall_ms": round(wall_ms, 3), "rays": int(st.rays), "launches": int(st.launches),
                         "grays_s": round(st.rays / ms / 1e6, 3)}
        rec["aov_over_render"] = round(rec["aov"]["ms"] / rec["render"]["ms"], 4)
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
