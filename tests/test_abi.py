"""The C-ABI library loads, exports every symbol include/rt1w.h declares, and fails loudly without a GPU."""
import ctypes as C
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "rt1w.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rt1w_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(rt):
    lib = rt.api.load_library()
    names = _declared_symbols()
    assert set(names) == set(rt.api.ABI_SYMBOLS), "api.ABI_SYMBOLS out of date with include/rt1w.h"
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/rt1w.h but not exported by librt1w.so"
    assert lib.rt1w_abi_version() == 2


def test_host_library_exports(rt):
    h = rt.api.load_host_library()
    text = open(os.path.join(ROOT, "raytracing-1w_b200", "host", "host_api.h")).read()
    for name in set(re.findall(r"\b(rt1w_host_[a-z0-9_]+)\s*\(", text)):
        assert hasattr(h, name)


def test_struct_layouts_match_the_header(rt):
    """ctypes mirrors vs the C compiler's view of include/rt1w.h (sizes probed through a tiny C program)."""
    import subprocess
    import tempfile

    api = rt.api
    src = r'''
#include <stdio.h>
#include "rt1w.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(rt1w_node), sizeof(rt1w_material), sizeof(rt1w_texture),
         sizeof(rt1w_perlin), sizeof(rt1w_image), sizeof(rt1w_scene_desc), sizeof(rt1w_camera), sizeof(rt1w_render_params),
         sizeof(rt1w_render_stats), sizeof(rt1w_scene_info), sizeof(rt1w_flat_prim), sizeof(rt1w_ray));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "p"), os.path.join(d, "p.c")])
        sizes = [int(x) for x in subprocess.check_output([os.path.join(d, "p")]).split()]
    mirrors = [api.Node, api.Material, api.Texture, api.Perlin, api.Image, api.SceneDesc, api.Camera, api.RenderParams,
               api.RenderStats, api.SceneInfo, api.FlatPrim, api.Ray]
    assert sizes == [C.sizeof(m) for m in mirrors]


# a child process with this environment sees no CUDA device, so the no-GPU checks below also run on a machine with GPUs
NO_GPU_ENV = dict(os.environ, CUDA_VISIBLE_DEVICES="")


def _context_statuses_without_a_gpu(*device_args):
    """The status of api.Context(a) for each argument, in a child process that sees no CUDA device."""
    import subprocess
    import sys

    code = ("import importlib, sys\n"
            f"sys.path.insert(0, {ROOT!r})\n"
            "api = importlib.import_module('raytracing-1w_b200').api\n"
            f"for a in {list(device_args)!r}:\n"
            "    try:\n"
            "        api.Context(a).close()\n"
            "        print(api.OK)\n"
            "    except api.Rt1wError as e:\n"
            "        print(e.status)\n")
    out = subprocess.check_output([sys.executable, "-c", code], env=NO_GPU_ENV, text=True, timeout=120)
    return [int(x) for x in out.split()]


def test_no_cpu_fallback(rt):
    """Without a usable CUDA device the product refuses to run (there is no CPU path to fall back to)."""
    assert _context_statuses_without_a_gpu(0) == [rt.api.ERR_NO_DEVICE]


def test_product_does_not_link_the_oracle(rt):
    """The shipped library must not depend on the checker."""
    import subprocess

    out = subprocess.check_output(["ldd", rt.api.LIB_PATH], text=True)
    assert "oracle" not in out
    syms = subprocess.check_output(["nm", "-D", "--defined-only", rt.api.LIB_PATH], text=True)
    assert "oracle_" not in syms


def test_demo_driver_fails_loudly_without_a_gpu(rt):
    """rt1w_main (the reference's `main` on top of the C ABI) exists and has no CPU path either."""
    import subprocess

    exe = os.path.join(os.path.dirname(rt.api.LIB_PATH), "rt1w_main")
    assert os.path.exists(exe)
    r = subprocess.run([exe, "cornel_box", "--width", "8", "--spp", "1"], capture_output=True, text=True, timeout=60, env=NO_GPU_ENV)
    assert r.returncode == 1 and "rt1w_context_create" in r.stderr
    assert not r.stdout.startswith("P3")


def test_library_shard_rule_matches_the_host_side(rt):
    """rt1w_shard_sample_range (what a communicator's ranks render) == shard.sample_range (host-side rule): a partition of
    the sample range into contiguous parts whose sizes differ by at most one."""
    import importlib

    shard = importlib.import_module("raytracing-1w_b200.shard")
    for world in (1, 2, 3, 4, 8):
        for begin, end in ((0, 1), (0, 7), (0, 100), (0, 4096), (300, 400), (5, 6)):
            ranges = [rt.api.shard_sample_range(r, world, begin, end) for r in range(world)]
            assert ranges[0][0] == begin and ranges[-1][1] == end
            assert all(ranges[i][1] == ranges[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in ranges]
            assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 0
            assert [(a - begin, b - begin) for a, b in ranges] == [shard.sample_range(r, world, end - begin) for r in range(world)]


def test_multi_gpu_entry_points_fail_loudly_without_a_gpu(rt):
    assert _context_statuses_without_a_gpu([0, 1], []) == [rt.api.ERR_NO_DEVICE, rt.api.ERR_INVALID]


def _c_prototypes():
    """name -> number of parameters, from include/rt1w.h."""
    text = open(os.path.join(ROOT, "include", "rt1w.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = {}
    for name, args in re.findall(r"\b(rt1w_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        args = args.strip()
        out[name] = 0 if args in ("", "void") else args.count(",") + 1
    return out


def test_rust_shim_declares_the_whole_abi():
    """The reference-side binding (rust/src/ffi.rs - source only, no Rust toolchain in this image) and the `extern "C"` block
    of INTEGRATION.md stay in step with include/rt1w.h: every exported function is declared in ffi.rs with the same number
    of parameters, every struct of the header has a #[repr(C)] mirror with the same number of fields, and INTEGRATION.md
    names no function the header does not have."""
    protos = _c_prototypes()
    assert set(protos) == set(_declared_symbols())
    rs = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    rs = re.sub(r"//[^\n]*", "", rs)
    decl = {}
    for name, args in re.findall(r"pub fn (rt1w_[a-z0-9_]+)\s*\(([^)]*)\)", rs, flags=re.S):
        args = args.strip().rstrip(",")
        decl[name] = 0 if not args else args.count(",") + 1
    missing = sorted(set(protos) - set(decl))
    assert not missing, f"rust/src/ffi.rs lacks {missing}"
    assert not sorted(set(decl) - set(protos)), "rust/src/ffi.rs declares functions the header does not have"
    wrong = {n: (protos[n], decl[n]) for n in protos if protos[n] != decl[n]}
    assert not wrong, f"parameter counts differ (header, ffi.rs): {wrong}"
    # structs: field counts
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rt1w.h")).read(), flags=re.S)
    for name, body in re.findall(r"typedef struct (rt1w_[a-z0-9_]+) \{(.*?)\} \1;", hdr, flags=re.S):
        c_fields = sum(len(decl_.split(",")) for decl_ in body.split(";") if decl_.strip())
        m = re.search(r"pub struct %s \{(.*?)\n\}" % name, rs, flags=re.S)
        assert m, f"rust/src/ffi.rs has no mirror of {name}"
        assert len(re.findall(r"pub [a-z0-9_]+\s*:", m.group(1))) == c_fields, f"{name}: field count differs from the header"
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert set(re.findall(r"\b(rt1w_[a-z0-9_]+)\s*\(", doc)) - {"rt1w_main"} <= set(protos) | {"rt1w_check"}
