"""PNG files encoded on the device (rtrb_encode_png / rtrb_submit_png, Camera.render_png): every file is taken apart
chunk by chunk, inflated with zlib and decoded with PIL, and must hold exactly the RGB8 frame rtrb_render returns."""
import io
import struct
import zlib

import numpy as np
import pytest

from raytracing_rb_b200 import Camera, Renderer, World, _abi, make_opts, png_max_bytes, render_multi, scenes
from raytracing_rb_b200._lib import RtrbError

pytestmark = pytest.mark.gpu


def parse_png(data):
    """-> (IHDR fields, filtered scanlines).  Checks the signature, every chunk's CRC, IEND last, and that the IDAT
    payload is one complete zlib stream (which also checks its Adler-32)."""
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, chunks = 8, []
    while pos < len(data):
        n, = struct.unpack(">I", data[pos:pos + 4])
        tag, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert crc == zlib.crc32(tag + body) & 0xFFFFFFFF, (tag, pos)
        chunks.append((tag, body))
        pos += 12 + n
    assert pos == len(data)
    assert chunks[0][0] == b"IHDR" and chunks[-1] == (b"IEND", b"")
    assert {t for t, _ in chunks} == {b"IHDR", b"IDAT", b"IEND"}
    d = zlib.decompressobj()
    filtered = d.decompress(b"".join(b for t, b in chunks if t == b"IDAT")) + d.flush()
    assert d.eof and d.unused_data == b""
    return struct.unpack(">IIBBBBB", chunks[0][1]), filtered


def check_png(data, rgb):
    """The file decodes to `rgb` (H, W, 3); returns the filtered stream."""
    from PIL import Image
    H, W = rgb.shape[:2]
    ihdr, filtered = parse_png(data)
    assert ihdr == (W, H, 8, 2, 0, 0, 0)
    assert len(filtered) == H * (3 * W + 1)
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGB")), rgb)
    return filtered


def min_sum_abs_filters(rgb):
    """Per-row filter type by the minimum sum of |signed byte| over the five PNG filters, ties to the lowest type."""
    H, W = rgb.shape[:2]
    x = rgb.reshape(H, 3 * W).astype(np.int16)
    b = np.vstack([np.zeros((1, 3 * W), np.int16), x[:-1]])
    a = np.hstack([np.zeros((H, 3), np.int16), x[:, :-3]])
    c = np.hstack([np.zeros((H, 3), np.int16), b[:, :-3]])
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    paeth = np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))
    sums = []
    for pred in (np.zeros_like(x), a, b, (a + b) // 2, paeth):
        v = (x - pred) % 256
        sums.append(np.where(v < 128, v, 256 - v).sum(axis=1))
    return np.argmin(np.stack(sums, axis=1), axis=1)


def scene(cid, width=None, height=None):
    wdoc, cdoc = scenes.build(cid)
    if width:
        cdoc = dict(cdoc, width=width, height=height)
    world = World(wdoc)
    return world, Camera(world, cdoc)


def rgb_frame(cam, seed=1):
    return cam.renderer().render(cam.camera_desc(), make_opts(seed=seed, pixel_format=_abi.FMT_RGB8),
                                 want_rgb=False, want_hit=False).rgba


def device_png(cam, seed=1, fmt=_abi.FMT_RGB8):
    r = cam.renderer()
    r.render_device(cam.camera_desc(), make_opts(seed=seed, pixel_format=fmt, skip_outputs=3))
    return r.encode_png(cam.width, cam.height, fmt)


@pytest.mark.parametrize("cid,w,h", [(1, None, None), (2, 160, 90), (3, 96, 54), (4, 64, 36), (6, 96, 54)])
def test_small_scenes_decode_to_the_frame(cid, w, h):
    _, cam = scene(cid, w, h)
    rgb = rgb_frame(cam)
    filtered = check_png(device_png(cam), rgb)
    rows = np.frombuffer(filtered, np.uint8).reshape(cam.height, 3 * cam.width + 1)
    assert np.array_equal(rows[:, 0], min_sum_abs_filters(rgb))


@pytest.mark.parametrize("cid,w,h", [(2, 1920, 1080), (3, 960, 540)])
def test_full_frames_decode_filter_choice_and_size(cid, w, h):
    """Filter bytes pinned to the min-sum-abs rule; the file at most 1.10 x zlib level 1 of the same filtered stream."""
    _, cam = scene(cid, w, h)
    rgb = rgb_frame(cam)
    png = device_png(cam)
    filtered = check_png(png, rgb)
    rows = np.frombuffer(filtered, np.uint8).reshape(h, 3 * w + 1)
    assert np.array_equal(rows[:, 0], min_sum_abs_filters(rgb))
    z1 = len(zlib.compress(filtered, 1))
    assert len(png) <= 1.10 * z1, (len(png), z1)


def test_empty_world_is_black():
    _, cdoc = scenes.build(2, width=320, height=180)
    world = World({"max_distance": 10000, "soft_shadow_exponent": 2, "lights": [], "world_objects": []})
    cam = Camera(world, cdoc)
    rgb = rgb_frame(cam)
    assert not rgb.any()
    png = device_png(cam)
    check_png(png, rgb)
    assert len(png) < 0.01 * 180 * (3 * 320 + 1)


@pytest.mark.parametrize("w,h", [(1, 1), (1, 37), (53, 1), (85, 128), (85, 256), (85, 129), (85, 257), (341, 32),
                                 (341, 64), (341, 33), (341, 65)])
def test_odd_sizes_and_segment_boundaries(w, h):
    """1x1, one column, one row, and filtered streams of exactly one and two segments (85 and 341 pixels make rows
    of 256 and 1024 bytes), plus one row more."""
    _, cam = scene(2, w, h)
    check_png(device_png(cam), rgb_frame(cam))


def test_same_bytes_every_way():
    """Encoding twice, from RGBA8 or RGB8, after render_device or from a pipeline of four frames in flight: same file."""
    import torch
    _, cam = scene(3, 200, 120)
    r, cd = cam.renderer(), cam.camera_desc()
    a = device_png(cam, seed=2)
    assert device_png(cam, seed=2) == a
    assert device_png(cam, seed=2, fmt=_abi.FMT_RGBA8) == a
    assert r.encode_png(200, 120, _abi.FMT_RGBA8) == a  # the framebuffer still holds that frame
    check_png(a, rgb_frame(cam, seed=2))
    cap = png_max_bytes(200, 120)
    bufs = [torch.zeros(cap, dtype=torch.uint8).pin_memory().numpy() for _ in range(4)]
    for fmt in (_abi.FMT_RGB8, _abi.FMT_RGBA8):
        tickets = [r.submit_png(cd, bufs[i], make_opts(seed=2, pixel_format=fmt)) for i in range(4)]
        for t in tickets:
            png, stats, code = r.wait_png(t)
            assert code == _abi.RTRB_OK and png == a
    # a zeroed opts struct is accepted (RGBA8, seed 0, STRICT)
    t = r.submit_png(cd, bufs[0], _abi.RenderOpts())
    png, _, _ = r.wait_png(t)
    check_png(png, r.render(cd, make_opts(seed=0, precision=_abi.PREC_STRICT, pixel_format=_abi.FMT_RGB8),
                            want_rgb=False, want_hit=False).rgba)


def test_incompressible_input_uses_stored_blocks():
    import torch
    g = torch.Generator(device="cuda").manual_seed(7)
    W, H = 700, 300
    noise = torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    _, cam = scene(2, 64, 36)
    r = cam.renderer()
    torch.cuda.synchronize()
    png = r.encode_png(W, H, _abi.FMT_RGB8, src=noise.data_ptr())
    check_png(png, noise.cpu().numpy())
    assert len(png) <= png_max_bytes(W, H)
    rgba = torch.cat([noise, torch.full((H, W, 1), 255, dtype=torch.uint8, device="cuda")], dim=2).contiguous()
    torch.cuda.synchronize()
    assert r.encode_png(W, H, _abi.FMT_RGBA8, src=rgba.data_ptr()) == png


def test_invalid_arguments():
    import ctypes as C
    import torch
    from raytracing_rb_b200._lib import lib
    _, cam = scene(2, 64, 36)
    r, cd = cam.renderer(), cam.camera_desc()
    r.render_device(cd, make_opts(pixel_format=_abi.FMT_RGB8))
    cap = png_max_bytes(64, 36)
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t()
    assert lib().rtrb_encode_png(r.handle, None, 64, 36, _abi.FMT_RGB8, None, out.ctypes.data, cap - 1,
                                 C.byref(n)) == _abi.RTRB_ERR_INVALID
    assert lib().rtrb_encode_png(r.handle, None, 64, 36, 7, None, out.ctypes.data, cap, C.byref(n)) == _abi.RTRB_ERR_INVALID
    with pytest.raises(RtrbError) as e:
        r.encode_png(64, 36, 7)
    assert e.value.code == _abi.RTRB_ERR_INVALID
    pinned = torch.zeros(cap, dtype=torch.uint8).pin_memory().numpy()
    for buf, opts in ((out, make_opts()), (pinned, make_opts(rgba_device_out=r.framebuffer_ptr(64, 36))),
                      (pinned, make_opts(pixel_format=_abi.FMT_PNG_RGB8)), (pinned, make_opts(pixel_format=9)),
                      (pinned[:cap - 1], make_opts())):
        with pytest.raises(RtrbError) as e:
            r.submit_png(cd, buf, opts)
        assert e.value.code == _abi.RTRB_ERR_INVALID
    t = r.submit_png(cd, pinned, make_opts(pixel_format=_abi.FMT_RGB8))  # the refusals left no frame in flight
    check_png(r.wait_png(t)[0], rgb_frame(cam))


def raising_camera():
    """The scene of test_first_bad_pixel_in_the_adaptive_pass: a 40x over-bright highlight that extra samples hit."""
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
    return Camera(w, cdoc)


def test_raised_frame_still_yields_its_png(tmp_path):
    import torch
    cam = raising_camera()
    r, cd = cam.renderer(), cam.camera_desc()
    want = r.render(cd, make_opts(seed=5, pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False)
    assert want.code == _abi.RTRB_ERR_RAISED
    buf = torch.zeros(png_max_bytes(96, 54), dtype=torch.uint8).pin_memory().numpy()
    png, stats, code = r.wait_png(r.submit_png(cd, buf, make_opts(seed=5, pixel_format=_abi.FMT_RGB8)))
    assert code == _abi.RTRB_ERR_RAISED and stats["status"] == want.stats["status"]
    check_png(png, want.rgba)
    path = tmp_path / "raised.png"
    with pytest.raises(RuntimeError, match="color greater than 1"):
        cam.render_png(str(path), seed=5)
    assert path.read_bytes() == png


def test_render_png_writes_the_file_and_leaves_the_canvas(tmp_path):
    _, cam = scene(2, 320, 180)
    canvas = cam.canvas.copy()
    path = tmp_path / "sub" / "image.png"
    stats = cam.render_png(str(path), seed=3)
    assert stats["status"] == 0 and np.array_equal(cam.canvas, canvas)
    check_png(path.read_bytes(), rgb_frame(cam, seed=3))


def test_multi_gpu_gather_then_encode():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _, cam = scene(2, 320, 180)
    single = device_png(cam)
    rs = [cam.renderer(d) for d in range(2)]
    render_multi(rs, cam.camera_desc(), make_opts(pixel_format=_abi.FMT_RGB8), want_rgb=False, want_hit=False)
    assert rs[0].encode_png(320, 180, _abi.FMT_RGB8) == single
