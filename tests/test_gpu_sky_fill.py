"""Sky-fill frames (rtrb_sky_fill): whole depth-1 FAST64 pinhole frames resolved in the thread trace only the tiles
outside each super-tile row's sky run, and store the runs' tiles from fill CTAs at the end of the grid.  Frames,
float RGB, hit ids and every counter must stay STRICT's bit for bit: the headline frame and an all-sky camera, sky rows
split by a sphere, sizes that are not multiples of the 32-pixel tile (and rows that are not 16-byte aligned), the three
pixel formats with and without the float RGB / hit-id outputs, pipelined frames, overlapping frames into one buffer and
a scene update; windows, tile splits and progressive passes (which keep the row-major grid) as well."""
import copy

import numpy as np
import pytest

from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Camera, Renderer, World, _abi, make_opts, scenes

from test_gpu_cull_tables import SHARED, assert_same, d1_camera, render
from test_gpu_sky_tiles import horizon_world

pytestmark = pytest.mark.gpu

FORMATS = {"rgba8": _abi.FMT_RGBA8, "rgb8": _abi.FMT_RGB8, "png_rgb8": _abi.FMT_PNG_RGB8}


def split_world():
    """A sphere high above the horizon: its mask cuts the sky tiles of its rows in two."""
    w = horizon_world(n=4)
    w["world_objects"].append(scenes.matte("high", [12.0, 0.5, 3.0], 1.0, (0.7, 0.7, 0.2)))
    return w


ALL_SKY = dict(front=[-1.0, 0.0, 1.0], up=[1.0, 0.0, 1.0])  # 45 degrees up, away from the light


def config2(**cam):
    w, c = scenes.build(2)
    return w, dict(c, **cam)


CASES = {
    "config2": config2(),
    "config2_all_sky": config2(**ALL_SKY),
    "split_sky": (split_world(), d1_camera(width=320, height=180)),
    "odd_size": (split_world(), d1_camera(width=203, height=77)),      # partial tiles on both edges
    "unaligned_rows": (split_world(), d1_camera(width=101, height=45)),  # W * 3 = 303: RGB8 rows start anywhere
    "tiny": (horizon_world(), d1_camera(width=7, height=5, up=[0.0, 0.0, -1.0])),
}


def render_fmt(w, cam, precision, fmt, outputs, detail=True):
    world = World(copy.deepcopy(w))
    c = Camera(world, copy.deepcopy(cam)).camera_desc()
    r = Renderer(world.to_scene_desc(), 0)
    skip = 0 if outputs else _abi.SKIP_RGB | _abi.SKIP_HIT
    f = r.render(c, make_opts(seed=3, precision=precision, count_detail=detail, pixel_format=FORMATS[fmt], skip_outputs=skip),
                 want_rgb=outputs, want_hit=outputs)
    r.close()
    return f


@pytest.mark.parametrize("case", sorted(CASES))
def test_fast_equals_strict(case):
    w, cam = CASES[case]
    for detail in (False, True):
        fast = render(w, cam, PREC_FAST64, detail)
        assert_same(fast, render(w, cam, PREC_STRICT, detail), case)
    if case == "config2_all_sky":
        assert (fast.hit < 0).all()
    if case in ("config2", "split_sky", "odd_size"):
        assert (fast.hit < 0).any() and (fast.hit >= 0).any()


@pytest.mark.parametrize("outputs", [True, False], ids=["rgb_hit", "bytes_only"])
@pytest.mark.parametrize("fmt", sorted(FORMATS))
@pytest.mark.parametrize("case", ["split_sky", "odd_size", "unaligned_rows"])
def test_pixel_formats(case, fmt, outputs):
    w, cam = CASES[case]
    for detail in (False, True):
        got = render_fmt(w, cam, PREC_FAST64, fmt, outputs, detail)
        want = render_fmt(w, cam, PREC_STRICT, fmt, outputs, detail)
        assert np.array_equal(got.rgba, want.rgba), (case, fmt)
        if outputs:
            assert np.array_equal(got.rgb, want.rgb) and np.array_equal(got.hit, want.hit), (case, fmt)
        assert {k: got.stats[k] for k in SHARED} == {k: want.stats[k] for k in SHARED}, (case, fmt)


def test_windows_tile_splits_and_progressive_passes():
    w, cam = CASES["split_sky"]
    world = World(copy.deepcopy(w))
    c = Camera(world, cam).camera_desc()
    r = Renderer(world.to_scene_desc(), 0)
    H, W = cam["height"], cam["width"]
    for opts in (dict(window=(5, 3, 250, 170)), dict(tile_rank=1, tile_world=3)):
        got, want = (r.render(c, make_opts(seed=3, precision=p, count_detail=True, **opts), out_rgba=np.zeros((H, W, 4), np.uint8))
                     for p in (PREC_FAST64, PREC_STRICT))
        assert np.array_equal(got.rgba, want.rgba) and got.rgba.any(), opts
        assert {k: got.stats[k] for k in SHARED} == {k: want.stats[k] for k in SHARED}, opts
    pcam = dict(cam, pre_sample_times=2, max_sample_times=2, variant_threshold=0.001)
    p = r.progressive(Camera(world, pcam).camera_desc(), make_opts(seed=3, precision=PREC_FAST64, count_detail=True))
    p.pass_to(2)
    got = p.download()
    p.close()
    want = r.render(Camera(world, pcam).camera_desc(), make_opts(seed=3, precision=PREC_STRICT, count_detail=True))
    r.close()
    assert np.array_equal(got.rgba, want.rgba) and np.array_equal(got.hit, want.hit) and np.array_equal(got.rgb, want.rgb)


def pitch_cams(world, cam, n):
    """A camera pitching from the ground through the horizon to the sky: the runs change every frame."""
    return [Camera(world, dict(cam, front=[1.0, 0.0, 0.35 * (k - n // 3)])).camera_desc() for k in range(n)]


def test_pipelined_frames_equal_strict():
    w, cam = CASES["split_sky"]
    world = World(copy.deepcopy(w))
    cams = pitch_cams(world, cam, 8)
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
        assert np.array_equal(bufs[k], r.render(c, make_opts(seed=3, precision=PREC_STRICT)).rgba), "frame %d" % k
    r.close()


def test_overlapping_frames_into_one_buffer():
    """Back-to-back frames into the renderer's framebuffer without a wait in between: the last frame's fill CTAs store
    after every write of the frame before, whose traced tiles are the last frame's sky."""
    w, cam = CASES["split_sky"]
    world = World(copy.deepcopy(w))
    r = Renderer(world.to_scene_desc(), 0)
    H, W = cam["height"], cam["width"]
    for order in ([0, 5], [5, 0], [0, 5, 2, 6, 1]):
        cams = pitch_cams(world, cam, 8)
        for k in order:
            r.render_device(cams[k], make_opts(seed=3, precision=PREC_FAST64), want_stats=False)
        rgba, rgb, hit = r.download(W, H)
        want = r.render(cams[order[-1]], make_opts(seed=3, precision=PREC_STRICT))
        assert np.array_equal(rgba, want.rgba) and np.array_equal(rgb, want.rgb) and np.array_equal(hit, want.hit), order
    r.close()


def test_scene_update_moving_a_sphere_into_the_sky():
    wa, cam = CASES["split_sky"]
    wb = copy.deepcopy(wa)
    wb["world_objects"][-1]["properties"]["center"] = [9.0, -2.0, 4.0]
    c = Camera(World(copy.deepcopy(wa)), copy.deepcopy(cam)).camera_desc()
    opts = make_opts(seed=1, precision=PREC_FAST64, count_detail=True)
    r = Renderer(World(copy.deepcopy(wa)).to_scene_desc(), 0)
    r.render(c, opts)
    r.update(World(copy.deepcopy(wb)).to_scene_desc())
    got = r.render(c, opts)
    r.close()
    want = render(wb, cam, PREC_STRICT)
    assert_same(got, want, "after the update")
