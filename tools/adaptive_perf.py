"""What adaptive sampling (rt1w_render_adaptive) saves against a uniform render, and what its sparse late rounds cost.

    python tools/adaptive_perf.py [--repeats R] [--out FILE]

Scenes at their bench sizes: C1 Cornell box 600x600, C3 final_scene 800x800.  Runs: uniform 1024 spp, and adaptive with
min_spp 16, cap 1024, max_error 0.5 / 1 / 2 levels.  Per run: ms per render (median of R after one warm-up), paths, rays,
rounds, and the error of the 8-bit image against a 4096-spp uniform reference rendered with another seed (RMSE and 99th
percentile of |difference|, in 8-bit levels).  Per round of the adaptive runs: the rate of that round alone, from the
difference of two renders whose caps are consecutive schedule steps (the rounds below the cap are the same renders).
Prints one JSON line per run; the GPU's name and power limit are read (a query only) and printed with them.
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

CONFIGS = [("C1", "cornel_box", 600, 600), ("C3", "final_scene", 800, 800)]
MIN_SPP, CAP, REF_SPP, ERRORS = 16, 1024, 4096, (0.5, 1.0, 2.0)


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True, timeout=30)
        return out.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def errors(rgb8, ref8):
    d = rgb8.astype(np.float64) - ref8.astype(np.float64)
    return float(np.sqrt(np.mean(d * d))), float(np.percentile(np.abs(d), 99))


def schedule(lo, hi):
    s = [lo]
    while s[-1] < hi:
        s.append(min(2 * s[-1], hi))
    return s


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

    def emit(rec):
        rec["gpu"] = info
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    for name, scene_name, w, h in CONFIGS:
        hs = api.HostScene(scene_name, seed=1)
        sc = api.Scene(ctx, hs.desc)
        cam = hs.camera()

        def params(spp, seed=0):
            return hs.params(width=w, height=h, spp=spp, seed=seed)

        ref8, _ = sc.render_rgb8(cam, params(REF_SPP, seed=0x5EED))

        def timed(fn):
            fn()  # warm-up
            runs = [fn() for _ in range(args.repeats)]
            return runs[-1], float(np.median([r[-1].render_ms for r in runs]))

        (rgb8, st), ms = timed(lambda: sc.render_rgb8(cam, params(CAP)))
        rmse, p99 = errors(rgb8, ref8)
        base_ms = ms
        emit({"config": name, "run": "uniform", "spp": CAP, "ms": round(ms, 2), "paths": int(st.paths), "rays": int(st.rays),
              "mpaths_s": round(st.paths / ms / 1e3, 1), "rmse_levels": round(rmse, 3), "p99_levels": round(p99, 2)})
        for err in ERRORS:
            (_, spp, rgb8, _, st), ms = timed(lambda: sc.render_adaptive(cam, params(CAP), MIN_SPP, err))
            rmse, p99 = errors(rgb8, ref8)
            steps = schedule(MIN_SPP, CAP)
            rounds = steps.index(int(spp.max())) + 1
            # per round: renders capped at consecutive schedule steps differ by exactly that round (+ its convergence pass)
            per_round, prev, prev_cap = None, None, 0
            per_round = []
            for cap in steps[:rounds]:
                sc.render_adaptive(cam, params(cap), MIN_SPP, err)  # warm-up at this cap
                r = [sc.render_adaptive(cam, params(cap), MIN_SPP, err)[-1] for _ in range(args.repeats)]
                cur = (float(np.median([x.render_ms for x in r])), int(r[-1].paths))
                d_ms, d_paths = (cur[0], cur[1]) if prev is None else (cur[0] - prev[0], cur[1] - prev[1])
                per_round.append({"samples": [prev_cap, cap], "pixels": d_paths // (cap - prev_cap), "ms": round(d_ms, 2),
                                  "mpaths_s": round(d_paths / d_ms / 1e3, 1) if d_ms > 0 else None})
                prev, prev_cap = cur, cap
            emit({"config": name, "run": "adaptive", "max_error": err, "min_spp": MIN_SPP, "cap": CAP, "ms": round(ms, 2),
                  "speedup_vs_uniform": round(base_ms / ms, 2), "paths": int(st.paths), "paths_vs_uniform": round(st.paths / (w * h * CAP), 3),
                  "rays": int(st.rays), "rounds": rounds, "mpaths_s": round(st.paths / ms / 1e3, 1), "rmse_levels": round(rmse, 3),
                  "p99_levels": round(p99, 2), "pixels_at_cap": int((spp == CAP).sum()), "per_round": per_round})
        sc.close()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
