"""Progressive frames (rtrb_progressive_*): after every pass the outputs (8-bit frame, float RGB compared as raw bits,
hit ids) and the stats equal rtrb_render_device's frame with pre = max = samples so far, and the final pass equals the
one-shot frame of the camera as given: configs 1 - 4, a BVH world, the box scene, STRICT and FAST64, every kind of
schedule; options, isolation from other work on the renderer, scene updates and argument errors."""
import ctypes as C

import numpy as np
import pytest

from raytracing_rb_b200 import Camera, World, _abi, make_opts, progressive_schedule, scenes, PREC_FAST64, PREC_STRICT
from raytracing_rb_b200._lib import RtrbError, check, lib
from raytracing_rb_b200.renderer import _frame_shape

pytestmark = pytest.mark.gpu

VOLATILE = ("exact_tests", "device_ms", "trace_ms")


def with_samples(cam, pre, mx):
    c = _abi.CameraDesc.from_buffer_copy(cam)
    c.pre_sample_times, c.max_sample_times = pre, mx
    return c


def oneshot(r, cam, opts):
    """rtrb_render_device + rtrb_download of the same outputs -> (frame bytes, rgb bits, hit, stats, code)."""
    stats, code = r.render_device(cam, opts)
    want_rgb = not (opts.skip_outputs & _abi.SKIP_RGB)
    want_hit = not (opts.skip_outputs & _abi.SKIP_HIT)
    fr = None if opts.rgba_device_out else np.empty(_frame_shape(cam.width, cam.height, opts.pixel_format), np.uint8)
    rgb = np.empty((cam.height, cam.width, 3), np.float64) if want_rgb else None
    hit = np.empty((cam.height, cam.width), np.int32) if want_hit else None
    check(lib().rtrb_download(r.handle, fr.ctypes.data if fr is not None else None, rgb.ctypes.data if want_rgb else None,
                              hit.ctypes.data if want_hit else None))
    return fr, rgb, hit, stats, code


def window_of(cam, opts):
    if opts.x1 == 0 and opts.y1 == 0:
        return 0, 0, cam.width, cam.height
    return opts.x0, opts.y0, opts.x1, opts.y1


def assert_same(got, want, cam, opts, what):
    """got: (Frame, stats, code) of a pass; want: oneshot().  Outside the window only the one-shot frame's stale
    framebuffer differs, so the outputs are compared on the window."""
    frame, stats, code = got
    fr, rgb, hit, wstats, wcode = want
    x0, y0, x1, y1 = window_of(cam, opts)
    assert code == wcode, what
    for k in wstats:
        if k not in VOLATILE:
            assert stats[k] == wstats[k], (what, k, stats[k], wstats[k])
    if fr is not None:
        if opts.pixel_format == _abi.FMT_PNG_RGB8:
            a, b = frame.rgba[y0:y1, 1 + 3 * x0:1 + 3 * x1], fr[y0:y1, 1 + 3 * x0:1 + 3 * x1]
        else:
            a, b = frame.rgba[y0:y1, x0:x1], fr[y0:y1, x0:x1]
        if opts.tile_world > 1:  # the rank's tiles only: compare where the hit ids say the rank rendered
            mask = hit[y0:y1, x0:x1] != -3
            a, b = a[mask], b[mask]
        assert np.array_equal(a, b), what
    if rgb is not None:
        a, b = frame.rgb[y0:y1, x0:x1].view(np.uint64), rgb[y0:y1, x0:x1].view(np.uint64)
        if opts.tile_world > 1:
            mask = hit[y0:y1, x0:x1] != -3
            a, b = a[mask], b[mask]
        assert np.array_equal(a, b), what
    if hit is not None:
        assert np.array_equal(frame.hit, hit), what


def run_schedule(r, cam, opts, sched, check_previews=True):
    pre = cam.pre_sample_times
    p = r.progressive(cam, opts)
    try:
        for e in sched:
            stats, code = p.pass_to(e)
            frame = p.download(not (opts.skip_outputs & _abi.SKIP_RGB), not (opts.skip_outputs & _abi.SKIP_HIT))
            if e < pre and not check_previews:
                continue
            ref_cam = cam if e == pre else with_samples(cam, e, e)
            assert_same((frame, stats, code), oneshot(r, ref_cam, opts), cam, opts, "pass to %d of %s" % (e, sched))
    finally:
        p.close()


def schedules(pre):
    out = [[pre], progressive_schedule(pre)]
    if pre > 1:
        out.append([1, pre])
    if pre <= 16:
        out.append(list(range(1, pre + 1)))
    if pre > 5:
        out.append([3, 5, pre])
    return out


def scene(name):
    if name == "c1":
        w, c = scenes.build(1)
    elif name == "c2":
        w, c = scenes.build(2, width=96, height=54)
    elif name == "c3":
        w, c = scenes.build(3, width=96, height=54)
    elif name == "c4":
        w, c = scenes.build(4, width=64, height=36)
    elif name == "bvh64":
        w, c = scenes.build(5, width=48, height=27, spp=64, grid=6)
    elif name == "boxes":
        w, c = scenes.build(6, width=96, height=54)
    world = World(w)
    return world, Camera(world, c)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4", "bvh64", "boxes"])
def test_previews_and_final_equal_oneshot_frames(name, precision):
    world, cam = scene(name)
    r = cam.renderer()
    cd = cam.camera_desc()
    if name == "bvh64":
        assert len(world.world_objects) > 34  # > 32 spheres: the BVH kernels
    for count_detail in (True, False):
        opts = make_opts(seed=3, precision=precision, count_detail=count_detail)
        for sched in schedules(cd.pre_sample_times):
            run_schedule(r, cd, opts, sched, check_previews=count_detail or sched == [1, cd.pre_sample_times])


def raising_world():
    lt = scenes.light([4, -7, 1.0], 0.0)
    lt["properties"].update(high_light_angle=12, high_light_rate=40)
    g = scenes.ground()
    sph = scenes.matte("a", (5, -0.8, 0.2), 1.2, (1, 0.5, 0.3))
    for o in (g, sph):
        o["properties"]["reflective_attenuation"] = [0.0, 0.0, 0.0]
    return World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [lt], "world_objects": [g, sph]})


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_raising_scene_status_and_first_bad_at_every_pass(precision):
    w = raising_world()
    _, cdoc = scenes.build(1)
    cdoc = dict(cdoc, width=96, height=54, pre_sample_times=8, max_sample_times=12, variant_threshold=0.0,
                trace_depth=3, monte_carlo_diffusion_times=1, aperture_radius=0.0)
    cam = Camera(w, cdoc)
    cd = cam.camera_desc()
    r = cam.renderer()
    opts = make_opts(seed=5, precision=precision, count_detail=True)
    p = r.progressive(cd, opts)
    try:
        for e in range(1, 9):
            stats, code = p.pass_to(e)
            ref = oneshot(r, cd if e == 8 else with_samples(cd, e, e), opts)
            assert (stats["status"], stats["first_bad_x"], stats["first_bad_y"], code) == \
                (ref[3]["status"], ref[3]["first_bad_x"], ref[3]["first_bad_y"], ref[4]), e
            assert_same((p.download(), stats, code), ref, cd, opts, "raising pass %d" % e)
    finally:
        p.close()
    assert code == _abi.RTRB_ERR_RAISED


OPTION_CASES = {
    "window": dict(window=(13, 7, 71, 40)),
    "rgb8": dict(pixel_format=_abi.FMT_RGB8),
    "png_rgb8": dict(pixel_format=_abi.FMT_PNG_RGB8, window=(5, 3, 90, 50)),
    "skip_rgb": dict(skip_outputs=_abi.SKIP_RGB),
    "skip_both": dict(skip_outputs=_abi.SKIP_RGB | _abi.SKIP_HIT, pixel_format=_abi.FMT_RGB8),
}


@pytest.mark.parametrize("case", sorted(OPTION_CASES))
@pytest.mark.parametrize("name", ["c1", "c3"])
def test_options(name, case):
    _, cam = scene(name)
    r = cam.renderer()
    cd = cam.camera_desc()
    opts = make_opts(seed=2, count_detail=True, **OPTION_CASES[case])
    run_schedule(r, cd, opts, progressive_schedule(cd.pre_sample_times))


@pytest.mark.parametrize("name", ["c1", "c4"])
def test_three_rank_tile_split(name):
    _, cam = scene(name)
    r = cam.renderer()
    cd = cam.camera_desc()
    for rank in range(3):
        opts = make_opts(seed=4, count_detail=True, tile_rank=rank, tile_world=3)
        run_schedule(r, cd, opts, progressive_schedule(cd.pre_sample_times))


def test_rgba_device_out_and_png_of_previews():
    import torch
    _, cam = scene("c1")
    r = cam.renderer()
    cd = cam.camera_desc()
    W, H = cd.width, cd.height
    out = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda:0")
    opts = make_opts(seed=6, pixel_format=_abi.FMT_RGB8, rgba_device_out=out.data_ptr())
    p = r.progressive(cd, opts)
    try:
        assert p.frame_ptr() == out.data_ptr()
        for e in progressive_schedule(cd.pre_sample_times):
            p.pass_to(e)
            png = r.encode_png(W, H, _abi.FMT_RGB8, src=p.frame_ptr())
            got = out.cpu().numpy()
            with pytest.raises(RtrbError):  # the 8-bit frame went to rgba_device_out
                check(lib().rtrb_progressive_download(p._h, np.empty(W * H * 3, np.uint8).ctypes.data, None, None))
            ref_cam = cd if e == cd.pre_sample_times else with_samples(cd, e, e)
            ref_opts = make_opts(seed=6, pixel_format=_abi.FMT_RGB8)
            fr, _, _, _, _ = oneshot(r, ref_cam, ref_opts)
            assert np.array_equal(got, fr), e
            assert png == r.encode_png(W, H, _abi.FMT_RGB8), e  # the matching one-shot frame, just rendered
    finally:
        p.close()


def test_isolation_from_other_work_on_the_renderer():
    """Between passes: a frame, a submit / wait pair, a trace_rays call and a second progressive frame.  Neither
    progressive frame's result changes, and neither do theirs."""
    _, cam = scene("c1")
    r = cam.renderer()
    cd, cd3 = cam.camera_desc(), Camera(cam.world, scenes.build(3, width=96, height=54)[1]).camera_desc()
    opts = make_opts(seed=7, count_detail=True)
    opts3 = make_opts(seed=8, count_detail=True)
    # alone
    ref_a = oneshot(r, cd, opts)
    ref_b = oneshot(r, cd3, opts3)
    ref_frame = r.render(cd3, opts3)
    rays = np.ascontiguousarray(r.camera_rays(cd, seed=7)[0][:4096])
    ref_rays = r.trace_rays(rays, trace_depth=4, mc=1, seed=7)
    pinned = np.empty((cd3.height, cd3.width, 4), np.uint8)
    a, b = r.progressive(cd, opts), r.progressive(cd3, opts3)
    try:
        sched_a = progressive_schedule(cd.pre_sample_times)  # [1, 2, 3]
        sched_b = [1, 2, 4]
        for k in range(3):
            sa, ca = a.pass_to(sched_a[k])
            frame = r.render(cd3, opts3)
            assert np.array_equal(frame.rgba, ref_frame.rgba) and np.array_equal(frame.rgb.view(np.uint64), ref_frame.rgb.view(np.uint64))
            sb, cb = b.pass_to(sched_b[k])
            t = r.submit(cd3, pinned, opts3)
            r.wait(t)
            assert np.array_equal(pinned, ref_frame.rgba)
            rgb, hit, _, _ = r.trace_rays(rays, trace_depth=4, mc=1, seed=7)
            assert np.array_equal(rgb.view(np.uint64), ref_rays[0].view(np.uint64)) and np.array_equal(hit, ref_rays[1])
        assert_same((a.download(), sa, ca), ref_a, cd, opts, "first progressive frame")
        assert_same((b.download(), sb, cb), ref_b, cd3, opts3, "second progressive frame")
    finally:
        a.close()
        b.close()


def test_scene_updates_between_passes():
    world, cam = scene("c1")
    r = cam.renderer()
    cd = cam.camera_desc()
    opts = make_opts(seed=9, count_detail=True)
    ref = oneshot(r, cd, opts)
    # a no-op update (the wrappers call update before every frame) leaves the frame valid
    p = r.progressive(cd, opts)
    try:
        p.pass_to(1)
        r.update(world.to_scene_desc())
        p.pass_to(2)
        r.update(world.to_scene_desc())
        stats, code = p.pass_to(cd.pre_sample_times)
        assert_same((p.download(), stats, code), ref, cd, opts, "final after no-op updates")
    finally:
        p.close()
    # a real update makes the next pass fail
    p = r.progressive(cd, opts)
    try:
        p.pass_to(1)
        w2 = scenes.build(1)[0]
        w2["lights"][0]["properties"]["position"] = [v + 0.5 for v in w2["lights"][0]["properties"]["position"]]
        r.update(World(w2).to_scene_desc())
        with pytest.raises(RtrbError) as e:
            p.pass_to(2)
        assert e.value.code == _abi.RTRB_ERR_INVALID and "scene changed" in str(e.value)
    finally:
        p.close()
    r.update(world.to_scene_desc())


def test_argument_errors():
    _, cam = scene("c1")
    r = cam.renderer()
    cd = cam.camera_desc()
    pre = cd.pre_sample_times
    p = r.progressive(cd, make_opts(seed=1))
    try:
        with pytest.raises(RtrbError) as e:  # before the first pass
            p.download()
        assert e.value.code == _abi.RTRB_ERR_INVALID
        for bad in (0, -1, pre + 1):
            with pytest.raises(RtrbError) as e:
                p.pass_to(bad)
            assert e.value.code == _abi.RTRB_ERR_INVALID, bad
        p.pass_to(2)
        with pytest.raises(RtrbError) as e:  # not past what is done
            p.pass_to(2)
        assert e.value.code == _abi.RTRB_ERR_INVALID
        p.pass_to(pre)
        with pytest.raises(RtrbError) as e:  # after the final pass
            p.pass_to(pre)
        assert e.value.code == _abi.RTRB_ERR_INVALID
    finally:
        p.close()
    with pytest.raises(RtrbError) as e:
        r.progressive(cd, make_opts(rng_mode=_abi.RNG_MT))
    assert e.value.code == _abi.RTRB_ERR_UNSUPPORTED
    p = r.progressive(cd, make_opts(skip_outputs=_abi.SKIP_RGB))
    try:
        p.pass_to(1)
        with pytest.raises(RtrbError):
            p.download(want_rgb=True)
    finally:
        p.close()


def test_camera_render_progressive_matches_render_frame_and_render_png(tmp_path):
    _, cam = scene("c1")
    ref = cam.render_frame(seed=1)
    ref_png = tmp_path / "ref.png"
    cam.render_png(str(ref_png), seed=1)
    out = tmp_path / "prog.png"
    done = []
    for e, frame in cam.render_progressive(str(out), seed=1):
        done.append(e)
        assert out.exists()
    assert done == progressive_schedule(cam.pre_sample_times)
    assert np.array_equal(frame.rgba, ref.rgba)
    assert np.array_equal(frame.rgb.view(np.uint64), ref.rgb.view(np.uint64))
    assert np.array_equal(frame.hit, ref.hit)
    assert out.read_bytes() == ref_png.read_bytes()


def test_camera_render_progressive_raises_after_the_final_pass():
    w = raising_world()
    _, cdoc = scenes.build(1)
    cdoc = dict(cdoc, width=96, height=54, pre_sample_times=4, max_sample_times=4, variant_threshold=0.0,
                trace_depth=3, monte_carlo_diffusion_times=1, aperture_radius=0.0)
    cam = Camera(w, cdoc)
    gen = cam.render_progressive(seed=5)
    assert [e for e, _ in zip((1, 2), gen)] == [1, 2]
    with pytest.raises(RuntimeError):
        for _ in gen:
            pass
