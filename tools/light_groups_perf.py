"""What splitting the sums into light groups (rt1w_render_light_groups) costs against rt1w_render on the same arguments.

    python tools/light_groups_perf.py [--repeats R] [--out FILE]

Cases: the Cornell box at config 1 (600^2 x 100 spp, 2 groups), final_scene 800^2 x 16 spp, the 10^6-sphere stress scene
1920x1080 x 8 spp (16 light nodes + the background: 17 groups, 13 MB of sums per 65 536-pixel tile) and the Cornell box at
3840x2160 x 4 spp.  Groups: api.light_groups_by_node (every emissive leaf node its own group, the background last).
Per case both calls are warmed up once, then run R times each, alternating; the median of the device time between each
call's CUDA events (render_ms: memset, waves, tail; the host copy of the sums is outside it) and Mpaths/s.  The two must
trace the same rays.  Prints one JSON line per case; the GPU's name, power limit and max SM clock are read (a query only)
in the same run and printed first and with every line.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [  # name, scene, constructor arguments, width, height, spp
    ("C1", "cornel_box", {}, 600, 600, 100), ("final_scene", "final_scene", {}, 800, 800, 16),
    ("stress", "stress", dict(stress_spheres=1_000_000), 1920, 1080, 8), ("cornel_4k", "cornel_box", {}, 3840, 2160, 4),
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
        groups = api.light_groups_by_node(hs.desc)
        calls = {"render": lambda: sc.render(cam, p)[2], "groups": lambda: sc.render_light_groups(cam, p, groups)[1]}
        for fn in calls.values():
            fn()  # warm-up
        ms = {k: [] for k in calls}
        rays = {}
        for _ in range(args.repeats):
            for k, fn in calls.items():
                st = fn()
                ms[k].append(st.render_ms)
                rays[k] = int(st.rays)
        paths = w * h * spp
        rec = {"case": name, "scene": scene_name, "width": w, "height": h, "spp": spp, "groups": groups.n_groups, "paths": paths,
               "rays": rays["render"], "same_rays": rays["render"] == rays["groups"]}
        for k in calls:
            med = float(np.median(ms[k]))
            rec[k] = {"ms": round(med, 3), "mpaths_s": round(paths / med / 1e3, 1), "ms_all": [round(x, 3) for x in ms[k]]}
        rec["groups_over_render"] = round(rec["groups"]["ms"] / rec["render"]["ms"], 4)
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
