"""Depth-1 frames with ground certificates (rtrb_ground_rows): on a certified ground tile whose candidate mask is empty
the camera ray goes straight to the exact test of the scene's one plane.  The FAST64 depth-1 kernels (lean and generic
builds, and the generic build's progressive pass kernels) must stay bit-identical to STRICT, every counter included, on
scenes built to stress the certificates: long sphere shadows from a light low over the horizon, a light almost straight
above, a tilted plane, two planes (no certificate), a camera below the plane, a max_distance that cuts through the
ground, rolled and upside-down cameras and a far horizon; in windows, tile splits, overlapping pipelined frames,
progressive passes and after a scene update that moves a sphere onto certified tiles."""
import copy

import numpy as np
import pytest

from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Camera, Renderer, World, make_opts, scenes

from test_gpu_cull_tables import SHARED, assert_same, d1_camera, render

pytestmark = pytest.mark.gpu


def ground_world(light=(5.0, -4.0, 4.0), max_distance=10000, n=10, plane=None, extra_plane=None):
    objs = [plane or scenes.ground()]
    if extra_plane:
        objs.append(extra_plane)
    rs = np.random.RandomState(n)
    for i in range(n):
        c = [float(rs.uniform(2, 12)), float(rs.uniform(-4, 4)), float(rs.uniform(-0.9, 0.2))]
        objs.append(scenes.matte("s%d" % i, c, float(rs.uniform(0.1, 0.5)), tuple(rs.uniform(0.3, 1, 3))))
    w = scenes._world(objs, [scenes.light(list(light), 0.0)])
    w["max_distance"] = max_distance
    return w


def tilted_plane():
    p = scenes.ground()
    p["properties"].update(point=[0.0, 0.0, -1.2], front=[0.15, -0.1, 1.0], up=[1.0, 0.0, -0.15])
    return p


def second_plane():
    p = scenes.ground()
    p["properties"].update(name="wall", point=[30.0, 0.0, 0.0], front=[-1.0, 0.0, 0.0], up=[0.0, 0.0, 1.0])
    return p


DOWN = d1_camera(front=[1.0, 0.0, -0.35])
CASES = {
    "low_light": (ground_world(light=(-2.0, 3.0, -0.7)), DOWN),
    "light_overhead": (ground_world(light=(4.0, 0.1, 9.0)), DOWN),
    "tilted_plane": (ground_world(plane=tilted_plane()), DOWN),
    "two_planes": (ground_world(extra_plane=second_plane()), DOWN),
    "below_the_plane": (ground_world(), d1_camera(position=[0.0, 0.0, -3.0], front=[1.0, 0.0, 0.4])),
    "max_distance_cut": (ground_world(max_distance=4.5), DOWN),
    "rolled": (ground_world(), d1_camera(front=[1.0, 0.0, -0.3], up=[0.0, 0.5, 1.0])),
    "upside_down": (ground_world(), d1_camera(front=[1.0, 0.0, -0.3], up=[0.0, 0.0, -1.0])),
    "far_horizon": (ground_world(), d1_camera(position=[0.0, 0.0, 40.0], front=[1.0, 0.0, -0.08])),
}


@pytest.mark.parametrize("light_radius", [0.0, 0.5], ids=["lean", "generic"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_ground_scenes_fast_equals_strict(case, light_radius):
    w, cam = CASES[case]
    w = copy.deepcopy(w)
    w["lights"][0]["properties"]["radius"] = light_radius
    for detail in (False, True):
        fast = render(w, cam, PREC_FAST64, detail)
        assert_same(fast, render(w, cam, PREC_STRICT, detail), case)
    assert (fast.hit == 0).any()  # the frame sees the ground


def test_headline_frame_counters_unchanged():
    """Config 2 at full size: STRICT's frame, and the FAST64 refine count of the frame before ground certificates."""
    w, cdoc = scenes.build(2)
    fast = render(w, cdoc, PREC_FAST64)
    assert_same(fast, render(w, cdoc, PREC_STRICT), "config 2")
    assert fast.stats["exact_tests"] == 1301633


@pytest.mark.parametrize("opts", [dict(window=(5, 3, 150, 70)), dict(tile_rank=2, tile_world=3)], ids=["window", "tile_split"])
def test_windows_and_tile_splits(opts):
    w, cam = CASES["low_light"]
    cam = dict(cam, width=200, height=120)
    world = World(copy.deepcopy(w))
    r = Renderer(world.to_scene_desc(), 0)
    c = Camera(world, cam).camera_desc()
    got, want = (r.render(c, make_opts(seed=3, precision=prec, count_detail=True, **opts), out_rgba=np.zeros((120, 200, 4), np.uint8))
                 for prec in (PREC_FAST64, PREC_STRICT))
    r.close()
    assert np.array_equal(got.rgba, want.rgba) and got.rgba.any()
    assert {k: got.stats[k] for k in SHARED} == {k: want.stats[k] for k in SHARED}
    if "window" in opts:
        x0, y0, x1, y1 = opts["window"]
        for a, b in ((got.rgb, want.rgb), (got.hit, want.hit)):
            assert np.array_equal(a[y0:y1, x0:x1], b[y0:y1, x0:x1])


def test_pipelined_frames_equal_strict():
    """Overlapping frames of a camera pitching down onto the ground (the certificates change every frame)."""
    w, cam = CASES["light_overhead"]
    world = World(copy.deepcopy(w))
    cams = [Camera(world, dict(cam, front=[1.0, 0.0, -0.1 * k])).camera_desc() for k in range(8)]
    r = Renderer(world.to_scene_desc(), 0)
    bufs = [np.empty((cam["height"], cam["width"], 4), np.uint8) for _ in cams]
    tickets = []
    for k, c in enumerate(cams):
        tickets.append(r.submit(c, bufs[k], make_opts(seed=3, precision=PREC_FAST64)))
        if len(tickets) > 3:
            r.wait(tickets[-4])
    for t in tickets[-3:]:
        r.wait(t)
    for k, c in enumerate(cams):
        want = r.render(c, make_opts(seed=3, precision=PREC_STRICT))
        assert np.array_equal(bufs[k], want.rgba), "frame %d" % k
    r.close()


def test_progressive_passes_equal_one_shot_frames():
    w, cam = CASES["low_light"]
    cam = dict(cam, pre_sample_times=4, max_sample_times=4, variant_threshold=0.001)
    world = World(copy.deepcopy(w))
    c = Camera(world, cam).camera_desc()
    r = Renderer(world.to_scene_desc(), 0)
    p = r.progressive(c, make_opts(seed=3, precision=PREC_FAST64, count_detail=True))
    for e in (1, 2, 4):
        p.pass_to(e)
        got = p.download()
        ce = Camera(world, dict(cam, pre_sample_times=e, max_sample_times=e)).camera_desc()
        want = r.render(ce, make_opts(seed=3, precision=PREC_STRICT, count_detail=True))
        assert np.array_equal(got.rgba, want.rgba) and np.array_equal(got.hit, want.hit), "pass to %d" % e
        assert np.array_equal(got.rgb, want.rgb), "pass to %d" % e
    p.close()
    r.close()


def test_update_moving_a_shadow_onto_certified_tiles():
    """A sphere moved into the camera's footprint: its tiles lose their empty mask, and its shadow falls on ground tiles."""
    wa, cdoc = CASES["light_overhead"]
    wb = copy.deepcopy(wa)
    wb["world_objects"][1]["properties"]["center"] = [3.0, 0.0, -0.6]
    wb["world_objects"][1]["properties"]["radius"] = 0.4
    cam = Camera(World(copy.deepcopy(wa)), copy.deepcopy(cdoc)).camera_desc()
    opts = make_opts(seed=1, precision=PREC_FAST64, count_detail=True)
    r = Renderer(World(copy.deepcopy(wa)).to_scene_desc(), 0)
    r.render(cam, opts)
    r.update(World(copy.deepcopy(wb)).to_scene_desc())
    got = r.render(cam, opts)
    r.close()
    assert_same(got, render(wb, cdoc, PREC_STRICT), "after the update")
