"""C-ABI contract details fixed in round 2 (ADVICE r1): where the 8-bit frame goes, when the framebuffer may move,
which ticket rtrb_wait accepts, and which pixel a raise is attributed to in the adaptive extra-sample pass."""
import numpy as np
import pytest

from helpers_rtrb import load_scene
from raytracing_rb_b200 import PREC_FAST64, PREC_STRICT, Renderer, _abi, make_opts
from raytracing_rb_b200._lib import RtrbError

pytestmark = pytest.mark.gpu


def test_host_buffer_calls_reject_rgba_device_out():
    """rtrb_render / rtrb_render_multi copy the renderer's own framebuffer to the host: with rgba_device_out the frame
    would be somewhere else and the host buffer stale, so they refuse (RTRB_ERR_INVALID), and rtrb_download refuses to
    hand out an 8-bit frame that was written elsewhere."""
    world, cam = load_scene(2, width=160, height=90)
    r, c = cam.renderer(), cam.camera_desc()
    other = Renderer(world.to_scene_desc(), 0)
    ptr = other.framebuffer_ptr(160, 90)
    with pytest.raises(RtrbError) as e:
        r.render(c, make_opts(rgba_device_out=ptr))
    assert e.value.code == _abi.RTRB_ERR_INVALID
    r.render_device(c, make_opts(rgba_device_out=ptr))      # the device-buffer call accepts it ...
    with pytest.raises(RtrbError):
        r.download(160, 90, want_rgb=False, want_hit=False)  # ... and the renderer's own framebuffer holds no frame
    want = r.render(c, make_opts(), want_rgb=False, want_hit=False).rgba
    got = np.zeros((90, 160, 4), np.uint8)
    other.framebuffer_download(160, 90, got)
    assert np.array_equal(got, want)


def test_exported_framebuffer_is_pinned():
    """Once its address or IPC handle is out, the framebuffer must not be reallocated under the peers' feet: a larger
    frame fails loudly instead (a smaller one keeps working in the same memory)."""
    world, cam = load_scene(2, width=64, height=36)
    r = Renderer(world.to_scene_desc(), 0)
    p1 = r.framebuffer_ptr(64, 36)
    assert r.framebuffer_ptr(32, 18) == p1
    with pytest.raises(RtrbError) as e:
        r.framebuffer_ptr(128, 72)
    assert e.value.code == _abi.RTRB_ERR_INVALID
    big = load_scene(2, width=128, height=72)[1].camera_desc()
    with pytest.raises(RtrbError):
        r.render(big, make_opts())
    small = r.render(cam.camera_desc(), make_opts(), want_rgb=False, want_hit=False)
    assert small.rgba.shape == (36, 64, 4) and r.framebuffer_ptr(64, 36) == p1


def test_wait_rejects_stale_and_duplicate_tickets():
    import torch
    world, cam = load_scene(2, width=64, height=36)
    r, c = cam.renderer(), cam.camera_desc()
    buf = torch.zeros((36, 64, 4), dtype=torch.uint8).pin_memory().numpy()
    t0 = r.submit(c, buf, make_opts())
    r.wait(t0)
    with pytest.raises(RtrbError):          # duplicate: already waited for
        r.wait(t0)
    tickets = [r.submit(c, buf, make_opts()) for _ in range(4)]
    with pytest.raises(RtrbError):          # stale: same slot (ticket % 4) as tickets[3], but not the frame in it
        r.wait(tickets[3] - 4)
    with pytest.raises(RtrbError):          # a fifth frame does not fit
        r.submit(c, buf, make_opts())
    for t in tickets:
        r.wait(t)


def test_framebuffer_copy_async_delivers_the_frame():
    import torch
    world, cam = load_scene(3, width=96, height=54)
    r, c = cam.renderer(), cam.camera_desc()
    want = r.render(c, make_opts(seed=3, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False).rgba
    host = torch.zeros((54, 96, 3), dtype=torch.uint8).pin_memory().numpy()
    s = torch.cuda.Stream()
    r.render_device(c, make_opts(seed=3, pixel_format=_abi.FMT_RGB8, stream=s.cuda_stream), want_stats=False)
    r.framebuffer_copy_async(96 * 54 * 3, host, s.cuda_stream)
    s.synchronize()
    assert np.array_equal(host, want)
    with pytest.raises(RtrbError):
        r.framebuffer_copy_async(1 << 30, host, s.cuda_stream)


@pytest.mark.parametrize("precision", [PREC_STRICT, PREC_FAST64])
def test_first_bad_pixel_in_the_adaptive_pass(oracle_mod, precision):
    """A raise that only happens in an EXTRA sample (camera.rb:88-93) must be attributed to the pixel it happened in,
    lowest x*H + y first, although the extra-sample kernel walks several pixels per thread."""
    from raytracing_rb_b200 import Camera, World, scenes
    # Matte, non-reflective ground and sphere; a point light far to the side whose highlight (world.rb:83-98) is 40x
    # over-bright.  Only the random Monte-Carlo rays spawned in the sphere's shadow (world_object.rb:76-90) can run
    # into the 12-degree highlight cone, so WHICH samples raise 'color greater than 1' is random per sample: with
    # pre = 1 and max = 12 the first offending pixel (0, 33) raises in an extra sample only (the oracle with
    # pre = max = 1 first raises at (3, 39)).
    lt = scenes.light([4, -7, 1.0], 0.0)
    lt["properties"].update(high_light_angle=12, high_light_rate=40)
    g = scenes.ground()
    sph = scenes.matte("a", (5, -0.8, 0.2), 1.2, (1, 0.5, 0.3))
    for o in (g, sph):
        o["properties"]["reflective_attenuation"] = [0.0, 0.0, 0.0]
    w = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [lt], "world_objects": [g, sph]})
    _, cdoc = scenes.build(1)
    cdoc = dict(cdoc, width=96, height=54, pre_sample_times=1, max_sample_times=12, variant_threshold=0.0,
                trace_depth=3, monte_carlo_diffusion_times=1, aperture_radius=0.0)
    cam = Camera(w, cdoc)
    sc = oracle_mod.OracleScene(w.to_scene_desc())
    ref = sc.render(cam.camera_desc(), make_opts(seed=5))
    pre_only = sc.render(Camera(w, dict(cdoc, max_sample_times=1)).camera_desc(), make_opts(seed=5))
    assert ref.stats["status"] & _abi.ST_COLOR_GT_1
    assert (ref.stats["first_bad_x"], ref.stats["first_bad_y"]) != (pre_only.stats["first_bad_x"], pre_only.stats["first_bad_y"]), \
        "the first offending pixel is meant to raise in an extra sample only"
    got = cam.render_frame(seed=5, precision=precision, count_detail=True)
    assert got.stats["status"] == ref.stats["status"]
    assert (got.stats["first_bad_x"], got.stats["first_bad_y"]) == (ref.stats["first_bad_x"], ref.stats["first_bad_y"])
    assert got.stats["adaptive_pixels"] == ref.stats["adaptive_pixels"] == 96 * 54
    assert got.stats["mc_rays"] == ref.stats["mc_rays"]
    assert np.array_equal(got.rgba, ref.rgba) and np.array_equal(got.hit, ref.hit)


@pytest.mark.parametrize("pre,mx,thr", [(4, 10, 0.001), (2, 8, 0.0), (8, 4, 0.0), (16, 16, 0.001), (3, 10, 0.001)])
def test_in_cta_resolve_equals_the_sample_buffer_path(oracle_mod, pre, mx, thr):
    """The FAST64 ray-tree kernels finish render_at inside the CTA when pre_sample_times divides the CTA size
    (RTRB_RESOLVE_IN_CTA; pre = 3 exercises the sample-buffer fallback); STRICT always goes through the sample buffer
    and resolve_kernel.  Both must give the oracle's frame: same adaptive pixels, same extra samples, same bytes."""
    from raytracing_rb_b200 import Camera, World, scenes
    wdoc, cdoc = scenes.build(1)
    cdoc = dict(cdoc, width=120, height=68, pre_sample_times=pre, max_sample_times=mx, variant_threshold=thr)
    world = World(wdoc)
    cam = Camera(world, cdoc)
    ref = oracle_mod.OracleScene(world.to_scene_desc()).render(cam.camera_desc(), make_opts(seed=2))
    a = cam.render_frame(seed=2, precision=PREC_STRICT, count_detail=True)
    b = cam.render_frame(seed=2, precision=PREC_FAST64, count_detail=True)
    assert np.array_equal(a.rgb, b.rgb) and np.array_equal(a.rgba, b.rgba) and np.array_equal(a.hit, b.hit)
    assert np.array_equal(b.rgba, ref.rgba) and np.array_equal(b.hit, ref.hit)
    for k in ("samples", "rays", "shadow_queries", "adaptive_pixels", "mc_rays"):
        assert a.stats[k] == b.stats[k] == ref.stats[k], k
    if thr == 0.0:
        assert b.stats["adaptive_pixels"] == 120 * 68


def test_png_scanline_format_is_idat_ready(tmp_path):
    """RTRB_FMT_PNG_RGB8: H scanlines of (filter byte 0, W x RGB8) - the stream Camera#save_image's encoder deflates
    (camera.rb:36-39).  Deflated and framed by the host, the file decodes to the RGB8 frame; blocking and pipelined."""
    import torch
    from PIL import Image
    from raytracing_rb_b200 import write_png_scanlines
    world, cam = load_scene(3, width=200, height=120)
    r, c = cam.renderer(), cam.camera_desc()
    rgb = r.render(c, make_opts(seed=4, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False).rgba
    rows = r.render(c, make_opts(seed=4, pixel_format=_abi.FMT_PNG_RGB8), want_rgb=False, want_hit=False).rgba
    assert rows.shape == (120, 200 * 3 + 1) and not rows[:, 0].any()
    assert np.array_equal(rows[:, 1:].reshape(120, 200, 3), rgb)
    path = tmp_path / "frame.png"
    write_png_scanlines(str(path), rows, 200, 120)
    assert np.array_equal(np.asarray(Image.open(path).convert("RGB")), rgb)
    buf = torch.full((120, 601), 7, dtype=torch.uint8).pin_memory().numpy()
    r.wait(r.submit(c, buf, make_opts(seed=4, pixel_format=_abi.FMT_PNG_RGB8)))
    assert np.array_equal(buf, rows)
