#!/usr/bin/env python
"""Headline benchmark: Mpaths/s of the Cornell box (main.rs scene 5: 600x600, 100 spp, depth 50) on N B200s.

    python bench.py --gpus 1 --steps K --warmup W              # the CUDA wavefront renderer (this repo)
    python bench.py --impl reference --steps K --warmup W      # the reference algorithm on the host CPU cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

--dump-outputs DIR  writes what the last timed headline step computed, as rt1w_render_device hands it to its caller:
        DIR/rgb_sum.npy, the per-pixel radiance sums of the whole sample range (float32, 600 x 600 x 3, 4.3 MB; NaN where
        a sample was NaN, which the image shows as black).  The scene, camera and seeds are fixed, so two builds give the
        same numbers up to the order of the fp32 additions into a pixel.

A "step" is one render of the whole image for one sample range (W*H*spp paths).  With N > 1 (torchrun, one process per
GPU) every rank joins the LIBRARY's communicator (rt1w_context_comm_init; the id travels over torch.distributed, the
only thing torch.distributed does here besides barriers): render calls become collective, the library shards the sample
range [0, 100 N) over the ranks (100 spp per GPU: weak scaling) and adds the partial radiance sums with ONE ncclReduce on
the render stream.  Prints ONE JSON line (rank 0).

value   device-resident: scene committed, result left in HBM, timed with CUDA events on the render stream
e2e     through the C ABI the reference-side host calls (rt1w_render): camera/params in, radiance sums copied
        back to a pinned HOST buffer on rank 0 inside the timed region (reduce included)
roofline  the wave kernel (scatter + closest hit + regroup, one launch per wave) against the measured HBM peak, on
        SURVEY.md section 8(d)'s algorithmic bytes (148 B per ray segment + 60 B per path); kernel time measured
        live with CUDA events around every launch (RT1W_FLAG_PROFILE pass).  `fp32`: the secondary figure of SURVEY 8(d),
        fp32 (+ fp64) flops per ray counted by ncu in the committed capture (profiles/r02_flops.json) x the rays counted
        live, against 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4 TFLOP/s
configs   the other BASELINE.json configurations on this GPU count, each with its own roofline and (N = 1) CPU baseline:
        C2 random_scene 1200x800, C3 final_scene 800x800, C5 the 1 M-sphere stress scene 1920x1080 - timed at a reduced
        sample count (128 / 128 / 64 spp per step: long enough for the ramp at the two ends of a render not to count), and the STRONG-scaling jobs: C4 (Cornell 3840x2160, 4096 spp in
        total, reduce of 99.5 MB inside the step), C1 (100 spp in total) and C5 (256 spp in total), the same job at every N
cpu_baseline  the C++ f64 restatement of the reference (oracle/, kind "port": the Rust crate cannot be built in
        this image) on the host cores, on a bounded sample of the same workload
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

SCENE = "cornel_box"
WIDTH, HEIGHT, SPP, DEPTH = 600, 600, 100, 50
# SURVEY.md section 8(d): algorithmic bytes of one ray segment in a wavefront with fp32 SoA queues
BYTES_PER_RAY = 148.0       # whole pipeline
BYTES_PER_PATH = 60.0       # generate write + accumulate
FP32_PEAK_TFLOPS = 74.4     # 148 SM x 128 lanes x 2 x 1.965 GHz (BASELINE.md section 2)
METRIC = "Mpaths/s (Cornell box 600x600, 100 spp per GPU, depth 50)"

# The other BASELINE.json configurations (SURVEY.md section 8d).  `spp`: samples per pixel of one timed step (the config's own
# count is `full_spp`); `cpu`: the bounded sample the CPU baseline renders (width, height, spp): the config's own image at BASELINE.md
# section 3's 16 / 8 / 4 spp, 8 - 25 s of work for the host cores each.
CONFIGS = [
    dict(name="C2", scene="random_scene", workload="random_scene (main.rs:192-295,816-827: ~485 spheres, 1 in 5 moving, aperture 0.1) 1200x800, depth 50",
         width=1200, height=800, spp=128, full_spp=500, cpu=(1200, 800, 16)),
    dict(name="C2w", scene="one_weekend", workload="One-Weekend flavour of config 2 (static spheres, fuzz U[0,0.5)) 1200x800, depth 50",
         width=1200, height=800, spp=128, full_spp=500, cpu=(1200, 800, 16)),
    dict(name="C3", scene="final_scene", workload="final_scene (main.rs:635-795,916-936: 400 boxes, media, Perlin, earth map, 1000-sphere cluster) 800x800, depth 50",
         width=800, height=800, spp=128, full_spp=10000, cpu=(800, 800, 8)),
    dict(name="C5", scene="stress", workload="stress scene (SURVEY.md 8d: 10^6 random spheres + 16 rectangle lights, device-built BVH) 1920x1080, depth 50",
         width=1920, height=1080, spp=64, full_spp=256, cpu=(1920, 1080, 4)),
]
# Strong scaling: a FIXED job split over the ranks by the library's shard rule (total spp)
STRONG = [
    dict(name="C4", scene="cornel_box", workload="Cornell box 3840x2160 (16:9 camera), 4096 spp in total over all GPUs, depth 50; reduce of 99.5 MB inside the step",
         width=3840, height=2160, spp=4096, aspect=3840.0 / 2160.0),
    dict(name="C1", scene="cornel_box", workload="Cornell box 600x600, 100 spp in total over all GPUs, depth 50", width=600, height=600, spp=100),
    dict(name="C5", scene="stress", workload="stress scene 1920x1080, 256 spp in total over all GPUs, depth 50", width=1920, height=1080, spp=256),
]


def committed_profile_numbers():
    """Per-config numbers taken from the committed ncu captures (profiles/r02_flops.json, made by tools/ncu_flops.py):
    fp32 / fp64 flops per ray and, for the headline kernel, DRAM bytes of one steady-state launch."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_flops.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 6 and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_sample(api, oracle_binding, hs, width, spp, aspect=None, height=None):
    """The oracle port on all host cores on a bounded sample of a config: -> cpu_baseline dict."""
    osc = oracle_binding.OracleScene(hs.desc)
    p = hs.params(width=width, height=height, spp=spp)
    _, _, ost = osc.render(hs.camera() if aspect is None else hs.camera(aspect=aspect), p, threads=0)
    osc.close()
    return {"value": ost.paths / ost.seconds / 1e6, "unit": "Mpaths/s", "cores": int(ost.threads), "kind": "port",
            "sample": f"{p.width}x{p.height} x {spp} spp ({ost.paths} paths) of the same scene, {ost.seconds:.1f} s",
            "mrays_per_s": ost.rays / ost.seconds / 1e6}


def run_reference(args):
    """The reference arm: the reference's own CPU algorithm (oracle port) on all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rt = importlib.import_module("raytracing-1w_b200")
    api = rt.api
    import oracle_binding  # the one place besides tests/smoke where bench.py runs the oracle: as the measured reference arm

    hs = api.HostScene(SCENE, seed=1)
    osc = oracle_binding.OracleScene(hs.desc)
    cam = hs.camera()
    spp = args.ref_spp
    total_s, paths, rays, threads = 0.0, 0, 0, 1
    for step in range(args.warmup + args.steps):
        p = hs.params(width=WIDTH, spp=(step + 1) * spp, sample_begin=step * spp)
        _, _, st = osc.render(cam, p, threads=0)
        if step >= args.warmup:
            total_s += st.seconds
            paths += st.paths
            rays += st.rays
            threads = st.threads
    value = paths / total_s / 1e6
    sample = f"{WIDTH}x{HEIGHT} x {spp} spp per step ({WIDTH * HEIGHT * spp} paths), depth {DEPTH}, all rows"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cornel_box 600x600 depth 50 (main.rs:395-512,867-894), bounded sample", "sample": sample},
        "mrays_per_s": rays / total_s / 1e6, "rays_per_path": rays / max(paths, 1),
        "cpu_baseline": {"value": value, "unit": "Mpaths/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-spp", type=int, default=8, help="samples per pixel of one reference-arm step")
    ap.add_argument("--cpu-spp", type=int, default=32, help="samples per pixel of the cpu_baseline sample")
    ap.add_argument("--pool", type=int, default=0, help="paths in flight (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only: skip the other BASELINE configs and the strong-scaling jobs")
    ap.add_argument("--c4-spp", type=int, default=4096, help="total samples per pixel of the C4 strong-scaling job")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the radiance sums of the last timed headline step to DIR/rgb_sum.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the renderer has no CPU fallback")
    torch.cuda.set_device(local)
    rt = importlib.import_module("raytracing-1w_b200")
    api = rt.api
    ctx = api.Context(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # the library's own communicator: rank 0 makes the id, torch.distributed carries it (plumbing), every rank joins
        uid = torch.tensor(list(api.comm_unique_id()) if rank == 0 else [0] * api.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
        dist.broadcast(uid, src=0)
        ctx.comm_init(bytes(uid.cpu().tolist()), world, rank)

    stream = torch.cuda.current_stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB of L2
    peak, which = measured_peaks()
    prof = committed_profile_numbers()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_stats(ms, st_sum):
        """max over ranks of the device time, sums of this step's paths / rays / launches"""
        t = torch.tensor([ms, float(st_sum[0]), float(st_sum[1]), float(st_sum[2])], dtype=torch.float64, device="cuda")
        if world > 1:
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            t[0] = tmax[0]
        return float(t[0]), float(t[1]), float(t[2]), float(t[3])

    def timed_steps(scene, cam, params, accum, steps, warmup):
        """`steps` collective renders of `params` (the library shards the sample range over the ranks), device-timed."""
        for _ in range(warmup):
            scene.render_device(cam, params, accum.data_ptr(), stream.cuda_stream)
        total_ms, acc = 0.0, [0, 0, 0]
        for _ in range(steps):
            flush.zero_()  # L2 flush between timed iterations (not timed)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            st = scene.render_device(cam, params, accum.data_ptr(), stream.cuda_stream)
            e1.record(stream)
            torch.cuda.synchronize()
            total_ms += e0.elapsed_time(e1)
            acc[0] += st.paths
            acc[1] += st.rays
            acc[2] += st.launches
        barrier()
        return reduce_stats(total_ms, acc)

    def roofline_of(scene, cam, params, accum, key):
        """RT1W_FLAG_PROFILE pass (collective like every render call; rank 0's numbers): CUDA events around every launch."""
        p = params
        p.flags |= api.FLAG_PROFILE
        stp = scene.render_device(cam, p, accum.data_ptr(), stream.cuda_stream)
        p.flags &= ~api.FLAG_PROFILE
        wave_ms, wave_n = stp.kernel_ms[0], max(stp.kernel_launches[0], 1)
        alg_bytes = BYTES_PER_RAY * stp.rays + BYTES_PER_PATH * stp.paths  # all launches of this rank's share of one render
        achieved = alg_bytes / (wave_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "k_wave", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": prof.get(key, {}).get("dram_bytes_per_launch"), "peak_source": which,
                "algorithmic_bytes_per_launch": alg_bytes / wave_n, "avg_launch_ms": wave_ms / wave_n, "launches": int(wave_n)}
        fl = prof.get(key)
        fp32 = None
        if fl and fl.get("fp32_flops_per_ray"):
            tf = fl["fp32_flops_per_ray"] * stp.rays / (wave_ms * 1e-3) / 1e12
            fp32 = {"bound": "fp32", "achieved": tf, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": tf / FP32_PEAK_TFLOPS,
                    "fp32_flops_per_ray": fl["fp32_flops_per_ray"], "fp64_flops_per_ray": fl.get("fp64_flops_per_ray"),
                    "source": "flops per ray counted by ncu (fadd + fmul + 2 ffma, predicated-on threads) in the committed capture "
                              + str(fl.get("capture")) + " x rays counted live"}
        return roof, fp32, stp

    # ------------------------------------------------------------------ headline: C1, 100 spp per GPU (weak scaling)
    hs = api.HostScene(SCENE, seed=1)
    scene = api.Scene(ctx, hs.desc)
    cam = hs.camera()
    n_pixels = WIDTH * HEIGHT
    accum = torch.empty(n_pixels * 3, dtype=torch.float32, device="cuda")
    host_out = torch.empty(n_pixels * 3, dtype=torch.float32).pin_memory()

    def params(flags=0):  # the whole job: [0, 100 N); the library gives rank r [100 r, 100 (r + 1))
        return hs.params(width=WIDTH, height=HEIGHT, spp=SPP * world, sample_begin=0, seed=0, flags=flags, pool_paths=args.pool)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, paths, rays, launches = timed_steps(scene, cam, params(), accum, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # rank 0 holds the reduced image; read before the profile pass below reuses `accum`
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "rgb_sum.npy"), accum.view(HEIGHT, WIDTH, 3).cpu().numpy())
    value = paths / (total_ms * 1e-3) / 1e6
    mrays = rays / (total_ms * 1e-3) / 1e6

    # ---- end-to-end arm (host buffers through the C ABI: rt1w_render, collective at N > 1, the image lands on rank 0)
    out_np = host_out.numpy() if rank == 0 else None
    for _ in range(2):
        scene.render_into(cam, params(), out_np)
    barrier()
    e2e_s = 0.0
    for _ in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        scene.render_into(cam, params(), out_np)
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = (n_pixels * SPP * world * args.steps) / float(te[0]) / 1e6

    # ---- per-kernel times + rooflines
    roofline, fp32, stp = roofline_of(scene, cam, params(), accum, "C1")
    kernels = {}
    ksum = sum(stp.kernel_ms)
    for k, name in enumerate(api.KERNEL_NAMES):
        if stp.kernel_launches[k]:
            kernels[name] = {"ms": round(stp.kernel_ms[k], 3), "launches": int(stp.kernel_launches[k]), "share": round(stp.kernel_ms[k] / ksum, 4)}
    roofline["traffic_note"] = ("ncu dram read+write of ONE steady-state launch of the committed capture; the per-launch "
                                "average on the left includes the small launches of the tail")
    roofline["note"] = ("148 B per ray segment + 60 B per path (SURVEY.md 8d) over all k_wave launches of one render; the kernel moves 160 B "
                        "per segment through HBM and is bound by instruction issue / latency, see DESIGN.md")
    roofline["fp32"] = fp32

    # ---- CPU baseline on the host cores (rank 0, N = 1 only): the oracle port on a bounded sample
    want_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    oracle_binding = None
    cpu = None
    if want_cpu:
        import oracle_binding  # checker used as the reported CPU baseline (never on the product path)

        cpu = cpu_sample(api, oracle_binding, hs, WIDTH, args.cpu_spp)
    info = scene.info()
    scene.close()

    # ------------------------------------------------------------------ the other configs and the strong-scaling jobs
    configs, strong = [], []
    if not args.no_configs:
        del accum
        built = {}

        def scene_for(name):
            if name not in built:
                t0 = time.perf_counter()
                h = api.HostScene(name, seed=1, **({"stress_spheres": 1_000_000} if name == "stress" else {}))
                t1 = time.perf_counter()
                s = api.Scene(ctx, h.desc)
                built[name] = (h, s, t1 - t0, time.perf_counter() - t1)
            return built[name]

        for c in CONFIGS:  # every rank renders its share of `spp * world` samples: the per-GPU work of the config's own rate
            h, s, host_s, commit_s = scene_for(c["scene"])
            camc = h.camera()
            buf = torch.empty(c["width"] * c["height"] * 3, dtype=torch.float32, device="cuda")
            pc = h.params(width=c["width"], height=c["height"], spp=c["spp"] * world, seed=0)
            ms, cp, cr, cl = timed_steps(s, camc, pc, buf, 3, 1)
            roof, f32, _ = roofline_of(s, camc, pc, buf, c["name"])
            roof["fp32"] = f32
            i = s.info()
            rec = {"name": c["name"], "workload": c["workload"], "image": [c["width"], c["height"]], "spp_per_gpu_timed": c["spp"],
                   "spp_of_the_config": c["full_spp"], "steps": 3, "ms_per_step": ms / 3, "mpaths_per_s": cp / ms / 1e3, "mrays_per_s": cr / ms / 1e3,
                   "rays_per_path": cr / max(cp, 1.0), "gpu_launches": int(cl), "prims": i.n_prims, "bvh_nodes": i.n_bvh_nodes,
                   "scene_build": {"host_scene_s": round(host_s, 3), "commit_s": round(commit_s, 3), "lower_and_bvh_ms": round(i.build_ms, 1),
                                   "upload_ms": round(i.upload_ms, 1)},
                   "roofline": roof}
            if want_cpu:
                rec["cpu_baseline"] = cpu_sample(api, oracle_binding, h, c["cpu"][0], c["cpu"][2], height=c["cpu"][1])
                rec["gpu_over_cpu"] = rec["mpaths_per_s"] / rec["cpu_baseline"]["value"]
            configs.append(rec)
            del buf
        for c in STRONG:  # the SAME job at every N
            h, s, _, _ = scene_for(c["scene"])
            camc = h.camera(aspect=c["aspect"]) if "aspect" in c else h.camera()
            spp = args.c4_spp if c["name"] == "C4" else c["spp"]
            buf = torch.empty(c["width"] * c["height"] * 3, dtype=torch.float32, device="cuda")
            pc = h.params(width=c["width"], height=c["height"], spp=spp, seed=0, pool_paths=(1 << 23) if c["name"] == "C4" else 0)
            s.render_device(camc, h.params(width=c["width"], height=c["height"], spp=world, seed=0, pool_paths=pc.pool_paths), buf.data_ptr(),
                            stream.cuda_stream)  # warm-up: queues and communicator buffers allocated outside the timed step
            ms, cp, cr, cl = timed_steps(s, camc, pc, buf, 1, 0)
            strong.append({"name": c["name"], "workload": c["workload"], "scaling": "strong", "total_spp": spp, "n_gpus": world, "steps": 1,
                           "ms_per_step": ms, "mpaths_per_s": cp / ms / 1e3, "mrays_per_s": cr / ms / 1e3, "gpu_launches": int(cl),
                           "reduce_bytes": c["width"] * c["height"] * 12 if world > 1 else 0})
            del buf
        for h, s, _, _ in built.values():
            s.close()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 intersection / f32 shading", "data": "synthetic",
            "config": {"workload": "cornel_box 600x600, 100 spp per GPU, depth 50 (main.rs:395-512,867-894; BASELINE.json configs[0])",
                       "sharding": (f"sample ranges inside the library (rt1w_context_comm_init): rank r renders [{SPP}r, {SPP}(r+1)); "
                                    f"ncclReduce of {n_pixels * 12} B on the render stream") if world > 1 else "single GPU",
                       "l2": "flushed between timed iterations (256 MiB memset)", "pool_paths": args.pool or (1 << 23),
                       "prims": info.n_prims, "bvh_nodes": info.n_bvh_nodes},
            "mrays_per_s": mrays, "rays_per_path": rays / max(paths, 1.0),
            "e2e": {"value": e2e_value, "unit": "Mpaths/s", "h2d_bytes_per_step": 312, "d2h_bytes_per_step": n_pixels * 12},
            "gpu_launches": int(launches), "kernels": kernels, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "configs": configs, "strong_scaling": strong,
        }
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
