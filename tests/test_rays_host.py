"""Host-side checks of the ray-level C ABI (rtrb_trace_rays, rtrb_intersect_rays, rtrb_camera_rays) and of the
oracle's ray entry points they are tested against: struct layouts, exports, no CPU fallback, a hand-derived known
answer, and the oracle's own trace of its lens rays against its frame."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from raytracing_rb_b200 import World, _abi, scenes
from helpers_rtrb import load_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "raytracing_rb_b200", "csrc"), "-j4", "-s", "all"])
    from raytracing_rb_b200 import _lib
    return _lib.lib()


def test_ray_struct_sizes_match_header(L, tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rtrb_b200.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu\\n",sizeof(rtrb_ray),sizeof(rtrb_ray_hit),sizeof(rtrb_ray_opts),'
                   'offsetof(rtrb_ray_hit,distance),offsetof(rtrb_ray_opts,stream));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    from raytracing_rb_b200 import RAY_HIT_DTYPE
    assert got == [C.sizeof(_abi.Ray), C.sizeof(_abi.RayHit), C.sizeof(_abi.RayOpts), _abi.RayHit.distance.offset,
                   _abi.RayOpts.stream.offset]
    assert got[0] == 48 and got[1] == 72 == RAY_HIT_DTYPE.itemsize


def test_ray_symbols_are_exported_abi_unchanged(L):
    from raytracing_rb_b200 import _lib
    for name in ("rtrb_trace_rays", "rtrb_intersect_rays", "rtrb_camera_rays"):
        assert name in _lib.EXPORTS and hasattr(L, name)
    assert L.rtrb_abi_version() == _abi.ABI_VERSION == 4


def test_ray_calls_without_a_device_fail_with_cuda_error(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    rays = np.array([[0, 0, 0, 1, 0, 0]], np.float64)
    rgb, hit, keys = np.zeros((1, 3)), np.zeros(1, np.int32), np.zeros((1, 2), np.uint32)
    hits = np.zeros(1, np.uint8).repeat(C.sizeof(_abi.RayHit))
    opts = _abi.RayOpts()
    opts.precision, opts.trace_depth, opts.seed = _abi.PREC_FAST64, 1, 1
    st = _abi.Stats()
    assert L.rtrb_trace_rays(None, C.byref(opts), 1, rays.ctypes.data, None, rgb.ctypes.data, hit.ctypes.data,
                             C.byref(st)) == _abi.RTRB_ERR_CUDA
    assert L.rtrb_intersect_rays(None, C.byref(opts), 1, rays.ctypes.data, hits.ctypes.data) == _abi.RTRB_ERR_CUDA
    _, cam = load_scene(2, width=8, height=4)
    out = np.zeros((32, 6))
    assert L.rtrb_camera_rays(None, C.byref(cam.camera_desc()), C.byref(opts), 0, 1, out.ctypes.data,
                              keys.ctypes.data) == _abi.RTRB_ERR_CUDA
    assert L.rtrb_trace_rays(None, C.byref(opts), 0, None, None, None, None, None) == _abi.RTRB_ERR_CUDA


def _oracle():
    import rays_oracle
    return rays_oracle


def test_oracle_trace_kat_lambert_plus_ambient():
    """One sphere (C = (5, 0, 0), R = 1), one point light at (0, 0, 5) outside the 3-degree highlight cone of the ray,
    trace_depth 1: the ray along +x through the centre hits p = (4, 0, 0) (:in, n = p - C = (-1, 0, 0)), the light is
    unoccluded (area 1, 1^2 / 1 light), so the colour is ambient + diffuse * color * (L - p)^.n^ = 0.01 + 0.6 * 4/sqrt(41)
    (world_object.rb:51-74, ray_tracer.rb:152).  At exactly normal incidence the refraction child's
    normalize(reflection + d) is the zero vector, so the reference raises there (world_object.rb:136) although the child
    is born dead: status ZERO_VECTOR at ray 0, colour still written.  A ray that misses gives black and hit id -1."""
    ro = _oracle()
    world = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [scenes.light([0, 0, 5], 0.0)],
                   "world_objects": [scenes.matte("s", [5, 0, 0], 1.0, (1, 1, 1))]})
    o = ro.RayOracle(world.to_scene_desc())
    rays = np.array([[0, 0, 0, 1, 0, 0], [0, 0, 0, 0, 1, 0]], np.float64)
    rgb, hit, st, code = o.trace_rays(rays, trace_depth=1)
    want = 0.01 + 0.6 * (4.0 / math.sqrt(41.0))
    assert rgb[0] == pytest.approx([want] * 3, rel=0, abs=1e-15)
    assert list(hit) == [0, -1] and list(rgb[1]) == [0.0, 0.0, 0.0]
    assert code == _abi.RTRB_ERR_RAISED and st["status"] == _abi.ST_ZERO_VECTOR
    assert (st["first_bad_x"], st["first_bad_y"]) == (0, 0)
    assert (st["samples"], st["rays"], st["hits"], st["shadow_queries"], st["sphere_tests"]) == (2, 2, 1, 1, 2)
    h = o.intersect_rays(rays)
    assert list(h["object"]) == [0, -1] and list(h["face"]) == [-1, -1]
    assert list(h["intersection"][0]) == [4.0, 0.0, 0.0] and h["distance"][0] == 4.0 and h["direction"][0] == 1
    assert list(h["delta"][0]) == [-1e-5, 0.0, 0.0]


def test_oracle_trace_of_lens_rays_is_its_frame(oracle_mod):
    """Tracing the oracle's own lens rays keyed (y * W + x, 0) gives rtrb_oracle_render's RGB for one sample."""
    ro = _oracle()
    world, cam = load_scene(1)
    cam.width, cam.height = 24, 14
    cam.pre_sample_times = cam.max_sample_times = 1
    cam.aperture_radius = 0.002
    desc = cam.camera_desc()
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(desc, None)
    rays, keys = [], []
    for y in range(desc.height):
        for x in range(desc.width):
            pixel = y * desc.width + x
            a, b = oracle_mod.philox(1, 0, [pixel, 0, 0, 0])[:2]
            theta = ((a >> 5) * 67108864.0 + (b >> 6)) * (1.0 / 9007199254740992.0)
            front, pos = oracle_mod.lens_ray(desc, x, y, theta)
            rays.append(pos + front)
            keys.append((pixel, 0))
    rgb, hit, st, _ = ro.RayOracle(world.to_scene_desc()).trace_rays(
        np.array(rays), desc.trace_depth, desc.monte_carlo_diffusion_times, 1, np.array(keys))
    assert np.array_equal(rgb.reshape(ref.rgb.shape), ref.rgb)
    assert np.array_equal(hit.reshape(ref.hit.shape), ref.hit)
    assert st["rays"] == ref.stats["rays"] and st["mc_rays"] == ref.stats["mc_rays"]
