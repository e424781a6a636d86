"""Depth-1 frames with tile certificates (rtrb_tile_rows): sky tiles are stored without tracing and certified rows skip
the highlight test.  The FAST64 depth-1 kernels (lean and generic builds, and the generic build's progressive pass
kernels) must stay bit-identical to STRICT on scenes built to stress the certificates: the horizon crossing tiles at an
angle, the light inside the frame near the horizon, a far-plane cutoff at max_distance, a camera below the plane, in
windows, tile splits, overlapping pipelined frames, progressive passes and after a scene update."""
import copy

import numpy as np
import pytest

from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Camera, Renderer, World, make_opts, scenes

from test_gpu_cull_tables import SHARED, assert_same, d1_camera, render

pytestmark = pytest.mark.gpu


def horizon_world(light=(5.0, -4.0, 4.0), light_radius=0.0, max_distance=10000, n=8):
    objs = [scenes.ground()]
    rs = np.random.RandomState(n)
    for i in range(n):
        c = [float(rs.uniform(3, 14)), float(rs.uniform(-5, 5)), float(rs.uniform(-0.8, 1.2))]
        objs.append(scenes.matte("s%d" % i, c, float(rs.uniform(0.1, 0.6)), tuple(rs.uniform(0.3, 1, 3))))
    w = scenes._world(objs, [scenes.light(list(light), light_radius)])
    w["max_distance"] = max_distance
    return w


CASES = {
    "rolled_horizon": (horizon_world(), d1_camera(up=[0.0, 0.45, 1.0])),
    "light_near_horizon": (horizon_world(light=(12.0, 1.0, -0.6)), d1_camera()),
    "light_above_horizon": (horizon_world(light=(12.0, -2.0, 0.4)), d1_camera(up=[0.0, -0.2, 1.0])),
    "far_cutoff": (horizon_world(max_distance=9), d1_camera(front=[1.0, 0.0, -0.05])),
    "below_the_plane": (horizon_world(), d1_camera(position=[0.0, 0.0, -3.0], front=[1.0, 0.0, 0.3])),
    "upside_down": (horizon_world(), d1_camera(up=[0.0, 0.0, -1.0])),
    "depth_zero": (horizon_world(), d1_camera(trace_depth=0)),  # no certificates: the rays are not counted there
}


@pytest.mark.parametrize("light_radius", [0.0, 0.5], ids=["lean", "generic"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_certificate_scenes_fast_equals_strict(case, light_radius):
    w, cam = CASES[case]
    w = copy.deepcopy(w)
    w["lights"][0]["properties"]["radius"] = light_radius
    for detail in (False, True):
        fast = render(w, cam, PREC_FAST64, detail)
        assert_same(fast, render(w, cam, PREC_STRICT, detail), case)
    if case in ("rolled_horizon", "below_the_plane"):
        assert (fast.hit < 0).any() and (fast.hit >= 0).any()  # the frame has sky and ground


def test_headline_frame_full_size_fast_equals_strict():
    w, cdoc = scenes.build(2)
    assert_same(render(w, cdoc, PREC_FAST64), render(w, cdoc, PREC_STRICT), "config 2")


@pytest.mark.parametrize("opts", [dict(window=(5, 3, 150, 70)), dict(tile_rank=2, tile_world=3)], ids=["window", "tile_split"])
def test_windows_and_tile_splits(opts):
    """Only the pixels the frame renders are compared: the rest of the host buffers is never written."""
    w, cam = CASES["rolled_horizon"]
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
    """Overlapping frames of a camera pitching through the horizon (the certificates change every frame)."""
    w, cam = CASES["rolled_horizon"]
    world = World(copy.deepcopy(w))
    cams = [Camera(world, dict(cam, front=[1.0, 0.0, 0.15 * (k - 3)])).camera_desc() for k in range(8)]
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
    """The pass kernels take the sky path too: each pass equals the one-shot frame of its sample count."""
    w, cam = CASES["light_near_horizon"]
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


def test_update_moving_the_light_into_the_frame():
    wa, cdoc = CASES["rolled_horizon"]
    wb = copy.deepcopy(wa)
    wb["lights"][0]["properties"]["position"] = [12.0, 1.0, 0.5]
    cam = Camera(World(copy.deepcopy(wa)), copy.deepcopy(cdoc)).camera_desc()
    opts = make_opts(seed=1, precision=PREC_FAST64, count_detail=True)
    r = Renderer(World(copy.deepcopy(wa)).to_scene_desc(), 0)
    r.render(cam, opts)
    r.update(World(copy.deepcopy(wb)).to_scene_desc())
    got = r.render(cam, opts)
    r.close()
    assert_same(got, render(wb, cdoc, PREC_STRICT), "after the update")
