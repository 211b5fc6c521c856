"""Multi-GPU inside the library (SURVEY.md section 8e; include/rt1w.h "Multi-GPU"): a multi-device context shards the
sample range of every render call over its devices and adds the partial radiance sums with ncclReduce to the first one.

The N > 1 cases need a box with at least two GPUs (`gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`);
on a single-GPU box they are skipped and only the 1-device form of the same entry points runs."""
import os
import subprocess

import numpy as np
import pytest

from common import check_identical_render, check_identical_sums

pytestmark = pytest.mark.gpu


def _n_gpus():
    import torch

    return torch.cuda.device_count()


def test_one_device_multi_context_equals_plain_context(rt, gpu_ctx):
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    cam, p = hs.camera(), hs.params(width=64, spp=16, seed=7)
    plain = api.Scene(gpu_ctx, hs.desc)
    a = plain.render(cam, p)
    ctx = api.Context([0])
    assert ctx.comm() == (0, 1, 1)
    sc = api.Scene(ctx, hs.desc)
    b = sc.render(cam, p)
    check_identical_render(a, b, "one-device multi context", 16)  # (fp32 atomic sums: order varies from run to run)
    sc.close(), ctx.close(), plain.close()


@pytest.mark.parametrize("n", [2, 4, 8])
def test_n_devices_render_the_same_image(rt, gpu_ctx, n):
    """1 GPU and N GPUs: same paths, same rays, the same image up to the order of the fp32 additions; also with fewer
    samples than devices (some ranks only join the reduce), through every render entry point."""
    if _n_gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    api = rt.api
    hs = api.HostScene("cornel_box", seed=1)
    cam = hs.camera()
    one = api.Scene(gpu_ctx, hs.desc)
    ctx = api.Context(list(range(n)))
    assert ctx.comm() == (0, n, n)
    many = api.Scene(ctx, hs.desc)
    for spp in (32, n - 1, 1):
        p = hs.params(width=96, spp=spp, seed=11, flags=api.FLAG_STATS, stat_clamp=20.0)
        check_identical_render(one.render(cam, p, want_stat=True), many.render(cam, p, want_stat=True), f"{n} devices, {spp} spp", spp)
    p = hs.params(width=96, spp=32, seed=11)
    img_a, _ = one.render_rgb8(cam, p)
    img_b, _ = many.render_rgb8(cam, p)
    assert (np.abs(img_a.astype(int) - img_b.astype(int)) <= 1).all() and (img_a == img_b).mean() > 0.999
    many.close(), ctx.close(), one.close()


def test_demo_driver_on_two_gpus(rt):
    """rt1w_main --gpus 2 prints the same P3 image as on one GPU (8-bit levels, +-1 where the fp32 sums round differently)."""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    exe = os.path.join(os.path.dirname(rt.api.LIB_PATH), "rt1w_main")
    outs = []
    for gpus in (1, 2):
        r = subprocess.run([exe, "cornel_box", "--width", "48", "--spp", "16", "--gpus", str(gpus)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append(np.array(r.stdout.split()[4:], dtype=int))
    assert outs[0].shape == outs[1].shape and (np.abs(outs[0] - outs[1]) <= 1).all()


def _rank_worker(rank, world, uid, out_path):
    import importlib
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for q in (root, os.path.join(root, "tests")):
        if q not in sys.path:
            sys.path.insert(0, q)
    api = importlib.import_module("raytracing-1w_b200").api
    hs = api.HostScene("cornel_box", seed=1)
    ctx = api.Context(rank)
    ctx.comm_init(uid, world, rank)
    assert ctx.comm() == (rank, world, 1)
    sc = api.Scene(ctx, hs.desc)
    p = hs.params(width=96, spp=30, seed=11)
    out = np.empty((p.height, p.width, 3), np.float32) if rank == 0 else None
    st = sc.render_into(hs.camera(), p, out)
    lo, hi = api.shard_sample_range(rank, world, 0, 30)
    assert st.paths == 96 * 96 * (hi - lo)
    if rank == 0:
        np.save(out_path, out)
    sc.close(), ctx.close()


def test_one_process_per_gpu(rt, gpu_ctx, tmp_path):
    """The MPI / torchrun shape: rank 0 makes the id (rt1w_comm_unique_id), every process joins with
    rt1w_context_comm_init, rt1w_render is collective and rank 0 receives the image of the whole sample range."""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    api = rt.api
    uid = api.comm_unique_id()
    out_path = str(tmp_path / "img.npy")
    mp.get_context("spawn")
    mp.spawn(_rank_worker, args=(2, uid, out_path), nprocs=2, join=True)
    got = np.load(out_path)
    hs = api.HostScene("cornel_box", seed=1)
    one = api.Scene(gpu_ctx, hs.desc)
    ref, _, _ = one.render(hs.camera(), hs.params(width=96, spp=30, seed=11))
    check_identical_sums(got, ref, 30, "two ranks against one device")
    one.close()
