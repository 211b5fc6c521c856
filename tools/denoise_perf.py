"""What the denoiser (rt1w_denoise, rt1w_render_denoised) costs and what it buys.

    python tools/denoise_perf.py [--spp N] [--ref-spp M] [--repeats R] [--out FILE]

1. The filter alone at 600^2, 1920x1080 and 3840x2160 (synthetic sums, 5 passes): the device time of its kernels
   (torch.profiler, CUDA activities; prepare, the passes, finish and the rgb8 resolve) and the wall time of rt1w_denoise
   (which also uploads 17 floats per pixel from pageable host memory and copies the result back).
2. The six scenes of DESIGN.md section 13's table at their sizes, N spp (default 16), and the Cornell box at 3840x2160:
   rt1w_render_denoised (one call) against rt1w_render + rt1w_render_aov + rt1w_denoise on host buffers (the route without
   it), wall-clock medians of R calls after a warm-up, and the fused call's device time (render_ms); then RMSE in 8-bit
   levels of the noisy and the denoised image against an M-spp render with another seed (default 2048).
Prints one JSON line per case; the GPU's name, power limit and max SM clock are read (a query only) in the same run and
printed first and with every line.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

SIZES = [(600, 600), (1920, 1080), (3840, 2160)]
SCENES = [  # name, scene, constructor arguments, width, height
    ("C1", "cornel_box", {}, 600, 600), ("random_scene", "random_scene", {}, 1200, 800), ("one_weekend", "one_weekend", {}, 1200, 800),
    ("final_scene", "final_scene", {}, 800, 800), ("cornel_smoke", "cornel_smoke", {}, 600, 600),
    ("stress", "stress", dict(stress_spheres=1_000_000), 1920, 1080), ("C1_4k", "cornel_box", {}, 3840, 2160),
]


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True, timeout=30)
        return out.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError) as e:
        return f"unavailable ({e})"


def median_ms(fn, repeats):
    fn()  # warm-up
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        times.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(times))


def filter_kernel_ms(fn, repeats):
    """Device time of the filter's kernels per call, from a torch.profiler trace of `repeats` calls."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(repeats):
            fn()
    per = {}
    for ev in prof.key_averages():
        if "k_denoise" in ev.key or "k_resolve" in ev.key:
            key = next(k for k in ("prepare", "pass", "finish", "resolve") if k in ev.key)
            per[key] = per.get(key, 0.0) + ev.self_device_time_total / 1e3
    return {k: round(v / repeats, 4) for k, v in per.items()}, round(sum(per.values()) / repeats, 4)


def rmse(a8, b8):
    return round(float(np.sqrt(np.mean((a8.astype(np.float64) - b8) ** 2))), 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--ref-spp", type=int, default=2048)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from test_gpu_denoise import synthetic

    api = importlib.import_module("raytracing-1w_b200").api
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    ctx = api.Context(0)
    lines = []

    def emit(rec):
        rec["gpu"] = info
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    for w, h in SIZES:
        sums = synthetic(np.random.default_rng(1), h, w, args.spp)
        call = lambda: ctx.denoise(*sums, args.spp)
        per, total = filter_kernel_ms(call, args.repeats)
        bytes_in = 17 * 4 * w * h
        emit({"case": "filter", "width": w, "height": h, "passes": 5, "kernel_ms": total, "per_kernel_ms": per,
              "denoise_wall_ms": round(median_ms(call, args.repeats), 3), "host_input_mb": round(bytes_in / 2**20, 1)})

    for case, name, kw, w, h in SCENES:
        hs = api.HostScene(name, seed=1, **kw)
        sc = api.Scene(ctx, hs.desc)
        cam = hs.camera()
        p = hs.params(width=w, height=h, spp=args.spp, seed=1)
        ps = hs.params(width=w, height=h, spp=args.spp, seed=1, flags=api.FLAG_STATS)
        fused = lambda: sc.render_denoised(cam, p)
        fused_ms = median_ms(fused, args.repeats)

        def three():
            rgb_sum, stat, _ = sc.render(cam, ps, want_stat=True)
            aov = sc.render_aov(cam, p)[:4]
            return ctx.denoise(rgb_sum, stat, *aov, args.spp)

        three_ms = median_ms(three, args.repeats)
        _, den8, rgb_sum, _, st = sc.render_denoised(cam, p)
        render_ms = median_ms(lambda: sc.render(cam, ps, want_stat=True), args.repeats)
        rec = {"case": case, "scene": name, "width": w, "height": h, "spp": args.spp, "fused_wall_ms": round(fused_ms, 3),
               "three_calls_wall_ms": round(three_ms, 3), "render_stats_wall_ms": round(render_ms, 3),
               "fused_device_ms": round(st.render_ms, 3), "launches": int(st.launches)}
        if case != "C1_4k":
            ref8, _ = sc.render_rgb8(cam, hs.params(width=w, height=h, spp=args.ref_spp, seed=12345))
            rec.update({"ref_spp": args.ref_spp, "rmse_noisy": rmse(api.resolve_rgb8(rgb_sum, args.spp), ref8), "rmse_denoised": rmse(den8, ref8)})
        emit(rec)
        sc.close()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
