"""Depth-1 frames with the candidate masks (rtrb_cull_tables.h): the FAST64 depth-1 kernels (lean and generic builds)
must stay bit-identical to STRICT (RGBA8, float RGB, hit ids, status and first offending pixel) on scenes built to
stress the masks - the camera inside a sphere, spheres behind it, the light inside or on a sphere, spheres on the
light's cube-map edges, `up` not perpendicular to `front`, 1 and 31 spheres - on the bench's dolly frames, in windows
and tile splits, and after a scene update that moves the spheres and the light."""
import copy

import numpy as np
import pytest

from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Camera, Renderer, World, make_opts, scenes

pytestmark = pytest.mark.gpu

TIMINGS = ("device_ms", "trace_ms")
# what STRICT and FAST64 count alike (STRICT also counts the born-dead children of depth-1 frames and its stack depth)
SHARED = ("samples", "rays", "shadow_queries", "hits", "highlight_hits", "local_shaded", "lit_lights", "mc_rays",
          "texel_fetches", "adaptive_pixels", "status", "first_bad_x", "first_bad_y")


def d1_camera(**kw):
    cam = dict(scenes.COMMON_CAMERA, width=160, height=90, pre_sample_times=1, max_sample_times=1, trace_depth=1,
               monte_carlo_diffusion_times=0, aperture_radius=0.0)
    cam.update(kw)
    return cam


def stress_world(kind, light_radius):
    objs = [scenes.ground()]
    L = [5.0, -4.0, 4.0]
    if kind == "around_camera":
        objs.append(scenes.matte("around", [0.2, 0.0, 0.0], 1.0, (0.8, 0.5, 0.3)))
    if kind == "behind_camera":
        objs += [scenes.matte("b%d" % i, [-3.0 - i, -1.0 + i, -0.5], 0.6, (0.5, 0.5, 0.9)) for i in range(3)]
    if kind == "light_inside":
        objs.append(scenes.glass("light_shell", L, 0.7))
    if kind == "light_on_surface":
        objs.append(scenes.matte("touch_light", [L[0], L[1], L[2] - 0.5], 0.5, (0.9, 0.9, 0.9)))
    if kind == "cube_edges":  # centres along the diagonals of the light's cube map
        for i, d in enumerate(([1, 1, -1], [1, -1, -1], [-1, 1, -1], [1, 1, -0.5])):
            c = np.array(L) + 3.0 * np.array(d, float)
            objs.append(scenes.matte("edge%d" % i, [float(v) for v in c], 0.5, (0.6, 0.8, 0.6)))
    n = {"one": 1, "many": 31}.get(kind, 6)
    rs = np.random.RandomState(len(kind))
    for i in range(n):
        c = [float(rs.uniform(2.5, 12)), float(rs.uniform(-5, 5)), float(rs.uniform(-0.8, 1.5))]
        objs.append(scenes.matte("s%d" % i, c, float(rs.uniform(0.1, 0.7)), tuple(rs.uniform(0.3, 1, 3))))
    return scenes._world(objs, [scenes.light(L, light_radius)])


KINDS = ["around_camera", "behind_camera", "light_inside", "light_on_surface", "cube_edges", "one", "many"]


def render(world_doc, cam_doc, precision, count_detail=True, **opts):
    world = World(copy.deepcopy(world_doc))
    cam = Camera(world, copy.deepcopy(cam_doc)).camera_desc()
    r = Renderer(world.to_scene_desc(), 0)
    f = r.render(cam, make_opts(seed=3, precision=precision, count_detail=count_detail, **opts))
    r.close()
    return f


def assert_same(got, want, what="", vs_strict=True):
    """Frames, hit ids, status and the first offending pixel; against another FAST64 frame every counter as well."""
    assert np.array_equal(got.rgba, want.rgba), what + ": RGBA8"
    assert np.array_equal(got.rgb, want.rgb), what + ": float RGB"
    assert np.array_equal(got.hit, want.hit), what + ": hit ids"
    assert got.code == want.code, what
    keys = SHARED if vs_strict else [k for k in want.stats if k not in TIMINGS]
    assert {k: got.stats[k] for k in keys} == {k: want.stats[k] for k in keys}, what


@pytest.mark.parametrize("light_radius", [0.0, 0.5], ids=["lean", "generic"])
@pytest.mark.parametrize("kind", KINDS)
def test_stress_scenes_fast_equals_strict(kind, light_radius):
    w = stress_world(kind, light_radius)
    for cam in (d1_camera(), d1_camera(up=[0.3, 0.2, 1.0]), d1_camera(front=[1.0, 0.4, -0.3])):
        for detail in (False, True):  # the hot kernels and their full-counter variants
            assert_same(render(w, cam, PREC_FAST64, detail), render(w, cam, PREC_STRICT, detail), "%s %s" % (kind, cam["up"]))


@pytest.mark.parametrize("frame", [0, 31, 63])
def test_dolly_frames_fast_equals_strict(frame):
    w, cdoc = scenes.build(2, width=480, height=270)
    world = World(copy.deepcopy(w))
    cam = Camera(world, cdoc)
    c = cam.camera_desc()
    c.position[1] = c.position[1] + 0.02 * frame
    r = Renderer(world.to_scene_desc(), 0)
    a = r.render(c, make_opts(seed=1, precision=PREC_FAST64, count_detail=True))
    b = r.render(c, make_opts(seed=1, precision=PREC_STRICT, count_detail=True))
    r.close()
    assert_same(a, b, "dolly frame %d" % frame)


@pytest.mark.parametrize("opts", [dict(window=(37, 11, 141, 77)), dict(tile_rank=1, tile_world=3)],
                         ids=["window", "tile_split"])
def test_windows_and_tile_splits_fast_equals_strict(opts):
    w = stress_world("cube_edges", 0.0)
    cam = d1_camera(width=200, height=120)
    assert_same(render(w, cam, PREC_FAST64, **opts), render(w, cam, PREC_STRICT, **opts), str(opts))


def test_update_moving_spheres_and_light_equals_fresh_renderer():
    wa = stress_world("many", 0.0)
    wb = copy.deepcopy(wa)
    for o in wb["world_objects"]:
        if o["type"] == "Sphere":
            c = o["properties"]["center"]
            o["properties"]["center"] = [c[0] + 0.4, c[1] - 0.3, c[2]]
    wb["lights"][0]["properties"]["position"] = [3.0, 4.0, 6.0]
    cdoc = d1_camera()
    cam = Camera(World(copy.deepcopy(wa)), copy.deepcopy(cdoc)).camera_desc()
    opts = make_opts(seed=1, precision=PREC_FAST64, count_detail=True)
    r = Renderer(World(copy.deepcopy(wa)).to_scene_desc(), 0)
    r.render(cam, opts)
    r.update(World(copy.deepcopy(wb)).to_scene_desc())
    got = r.render(cam, opts)
    r.close()
    f = Renderer(World(copy.deepcopy(wb)).to_scene_desc(), 0)
    want = f.render(cam, opts)
    f.close()
    assert_same(got, want, "after the update", vs_strict=False)
    assert_same(got, render(wb, cdoc, PREC_STRICT, window=None), "against STRICT")
