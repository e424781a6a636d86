"""Animated PNG files encoded on the device (rtrb_apng_*, Renderer.apng, Camera.render_animation): every file is taken
apart chunk by chunk, every frame's rectangle is checked against numpy's bounding box of the changed pixels, every
frame's zlib stream against rtrb_encode_png of the same crop, and PIL's APNG reader must compose each frame exactly."""
import ctypes as C
import io
import struct
import zlib

import numpy as np
import pytest

from raytracing_rb_b200 import (Apng, Camera, Sphere, World, _abi, apng_frame_max_bytes, make_opts, png_max_bytes,
                                render_multi, scenes)
from raytracing_rb_b200._lib import RtrbError, lib
from raytracing_rb_b200.vec3 import Vec3

pytestmark = pytest.mark.gpu

RGB8 = _abi.FMT_RGB8


def parse_chunks(data):
    pos, out = 0, []
    while pos < len(data):
        n, = struct.unpack(">I", data[pos:pos + 4])
        tag, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert crc == zlib.crc32(tag + body) & 0xFFFFFFFF, (tag, pos)
        out.append((tag, body))
        pos += 12 + n
    assert pos == len(data)
    return out


def parse_apng(data, W, H):
    """-> list of frames {rect, fctl, chunks: data payloads (fdAT sequence numbers removed), tag}.  Checks the
    signature, every CRC, IHDR, acTL's frame count against the fcTL count, sequence numbers consecutive from 0 in file
    order, IEND last, and that every frame holds one complete zlib stream of h * (3w + 1) bytes."""
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    chunks = parse_chunks(data[8:])
    assert chunks[0][0] == b"IHDR" and struct.unpack(">IIBBBBB", chunks[0][1]) == (W, H, 8, 2, 0, 0, 0)
    assert chunks[1][0] == b"acTL" and chunks[-1] == (b"IEND", b"")
    num_frames, _ = struct.unpack(">II", chunks[1][1])
    frames, seq = [], 0
    for tag, body in chunks[2:-1]:
        if tag == b"fcTL":
            f = struct.unpack(">IIIIIHHBB", body)
            assert f[0] == seq
            seq += 1
            frames.append({"rect": (f[3], f[4], f[1], f[2]), "fctl": f[5:], "chunks": [], "tag": None})
            continue
        assert tag in (b"IDAT", b"fdAT") and frames
        fr = frames[-1]
        assert fr["tag"] in (None, tag)
        fr["tag"] = tag
        if tag == b"fdAT":
            assert struct.unpack(">I", body[:4])[0] == seq
            seq += 1
            body = body[4:]
        fr["chunks"].append(body)
    assert len(frames) == num_frames
    for k, fr in enumerate(frames):
        assert fr["tag"] == (b"IDAT" if k == 0 else b"fdAT")
        x0, y0, w, h = fr["rect"]
        assert 0 <= x0 and x0 + w <= W and 0 <= y0 and y0 + h <= H and w >= 1 and h >= 1
        d = zlib.decompressobj()
        raw = d.decompress(b"".join(fr["chunks"])) + d.flush()
        assert d.eof and d.unused_data == b"" and len(raw) == h * (3 * w + 1)
    return frames


def bbox(prev, cur):
    """(x0, y0, w, h) of the pixels whose RGB differs; 1 x 1 at (0, 0) when none does."""
    ys, xs = np.nonzero(np.any(prev != cur, axis=2))
    if len(xs) == 0:
        return (0, 0, 1, 1)
    return (int(xs.min()), int(ys.min()), int(xs.max() - xs.min() + 1), int(ys.max() - ys.min() + 1))


def idat_payloads(png):
    return [b for t, b in parse_chunks(png[8:]) if t == b"IDAT"]


def to_device(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check_file(data, frames_rgb, r, delay=(1, 25)):
    """`data` is an APNG of frames_rgb (list of H x W x 3): rectangles, streams against rtrb_encode_png, PIL decode."""
    import torch
    from PIL import Image
    H, W = frames_rgb[0].shape[:2]
    frames = parse_apng(data, W, H)
    assert len(frames) == len(frames_rgb)
    for k, fr in enumerate(frames):
        assert fr["fctl"] == (delay[0], delay[1], 0, 0)
        rect = (0, 0, W, H) if k == 0 else bbox(frames_rgb[k - 1], frames_rgb[k])
        assert fr["rect"] == rect, k
        x0, y0, w, h = rect
        crop = to_device(frames_rgb[k][y0:y0 + h, x0:x0 + w])
        torch.cuda.synchronize()
        assert fr["chunks"] == idat_payloads(r.encode_png(w, h, RGB8, src=crop.data_ptr())), k
    im = Image.open(io.BytesIO(data))
    assert getattr(im, "n_frames", 1) == len(frames_rgb)
    for k, want in enumerate(frames_rgb):
        im.seek(k)
        assert np.array_equal(np.asarray(im.convert("RGB")), want), k
    return frames


def apng_file(anim, chunks, plays=0):
    return anim.header(plays) + b"".join(chunks) + Apng.TRAILER


# ---- scenes --------------------------------------------------------------------------------------------------------
def config2(w=160, h=90):
    wdoc, cdoc = scenes.build(2, width=w, height=h)
    world = World(wdoc)
    return world, Camera(world, cdoc)


def sphere_index(world):
    return [i for i, o in enumerate(world.world_objects) if isinstance(o, Sphere)][0]


def move_sphere(world):
    """step(i) for config 2: one sphere moves every frame except frame 3."""
    k = sphere_index(world)

    def step(i):
        if i in (0, 3):
            return
        x, y, z = world.world_objects[k].center.to_a()
        world.world_objects[k].center = Vec3(x + 0.05, y - 0.04, z)
    return step


def blocking_animation(cam, step, n, seed=1, fmt=RGB8, between=None):
    """render + add, frame by frame -> (file, RGB8 frames, renderer)."""
    r = cam.renderer()
    anim = r.apng(cam.width, cam.height)
    chunks, rgbs = [], []
    for i in range(n):
        step(i)
        r = cam.renderer()
        cd = cam.camera_desc()
        rgbs.append(r.render(cd, make_opts(seed=seed, pixel_format=RGB8), want_rgb=False, want_hit=False).rgba)
        r.render(cd, make_opts(seed=seed, pixel_format=fmt), want_rgb=False, want_hit=False)
        if between:
            between(i)
        chunks.append(anim.add(pixel_format=fmt))
    data = apng_file(anim, chunks)
    anim.close()
    return data, rgbs, r


# ---- tests ---------------------------------------------------------------------------------------------------------
def test_moving_sphere_decodes_and_matches_the_standalone_encoder():
    world, cam = config2()
    data, rgbs, r = blocking_animation(cam, move_sphere(world), 12)
    frames = check_file(data, rgbs, r)
    assert frames[3]["rect"] == (0, 0, 1, 1)  # nothing moved before frame 3
    assert any(0 < f["rect"][2] * f["rect"][3] < 160 * 90 for f in frames[1:])
    # frame 0's IDAT chunks are rtrb_encode_png's for the same frame
    _, cam0 = config2()
    r0 = cam0.renderer()
    r0.render(cam0.camera_desc(), make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False)
    png0 = r0.encode_png(160, 90, RGB8)
    assert frames[0]["chunks"] == idat_payloads(png0)
    assert data[8 + 25 + 20:].startswith(b"\x00\x00\x00\x1afcTL")


def synthetic_frames(W, H, seed=3):
    """Random frame, then edits (XOR, so every edited byte changes): the last pixel, the last column, the last row,
    nothing, part of one row, the first column, the first pixel."""
    frames = [np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)]
    for region in ((H - 1, W - 1, 1), (slice(2, H - 3), W - 1, 0), (H - 1, slice(1, W - 4), 2), None,
                   (H // 2, slice(3, 9)), (slice(None), 0, 0), (0, 0, 2)):
        g = frames[-1].copy()
        if region is not None:
            g[region] ^= 0x55
        frames.append(g)
    return frames


def test_minimal_rectangles_and_formats():
    """Synthetic frames with changes at the canvas edges: the rectangles are the bounding boxes, and RGBA8, RGB8 and
    PNG_RGB8 sources give the same file."""
    import torch
    W, H = 83, 61
    rgbs = synthetic_frames(W, H)
    _, cam = config2(64, 36)
    r = cam.renderer()
    files = []
    for fmt in (_abi.FMT_RGB8, _abi.FMT_RGBA8, _abi.FMT_PNG_RGB8):
        anim = r.apng(W, H, delay=(3, 100))
        chunks = []
        for f in rgbs:
            if fmt == _abi.FMT_RGBA8:
                src = np.concatenate([f, np.full((H, W, 1), 255, np.uint8)], axis=2)
            elif fmt == _abi.FMT_PNG_RGB8:
                src = np.concatenate([np.zeros((H, 1), np.uint8), f.reshape(H, 3 * W)], axis=1)
            else:
                src = f
            t = to_device(src)
            torch.cuda.synchronize()
            chunks.append(anim.add(src=t.data_ptr(), pixel_format=fmt))
        assert anim.frames == len(rgbs)
        files.append(apng_file(anim, chunks))
        anim.close()
    assert files[1] == files[0] and files[2] == files[0]
    frames = check_file(files[0], rgbs, r, delay=(3, 100))
    assert [f["rect"] for f in frames[1:]] == [(W - 1, H - 1, 1, 1), (W - 1, 2, 1, H - 5), (1, H - 1, W - 5, 1),
                                                (0, 0, 1, 1), (3, H // 2, 6, 1), (0, 0, 1, H), (0, 0, 1, 1)]


def test_every_pixel_changes_4k_and_1x1():
    import torch
    _, cam = config2(64, 36)
    r = cam.renderer()
    g = torch.Generator(device="cuda").manual_seed(11)
    W, H = 3840, 2160
    noise = [torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]
    torch.cuda.synchronize()
    anim = r.apng(W, H)
    chunks = [anim.add(src=t.data_ptr()) for t in noise]
    rgbs = [t.cpu().numpy() for t in noise]
    frames = check_file(apng_file(anim, chunks), rgbs, r)
    assert all(f["rect"] == (0, 0, W, H) for f in frames)
    assert len(frames[1]["chunks"]) > 700  # hundreds of 32 KiB segments
    assert max(len(c) for c in chunks) <= apng_frame_max_bytes(W, H)
    anim.close()

    tiny = [np.array([[[v, 255 - v, 3]]], np.uint8) for v in (5, 5, 9, 200)]
    anim = r.apng(1, 1)
    chunks = []
    for f in tiny:
        t = to_device(f)
        torch.cuda.synchronize()
        chunks.append(anim.add(src=t.data_ptr()))
    frames = check_file(apng_file(anim, chunks), tiny, r)
    assert all(f["rect"] == (0, 0, 1, 1) for f in frames)
    anim.close()


def test_camera_fly_by_rectangles():
    world, cam = config2()
    x, y, z = cam.position.to_a()

    def step(i):
        cam.position = Vec3(x, y + 0.1 * i, z + 0.02 * i)
    data, rgbs, r = blocking_animation(cam, step, 5)
    frames = check_file(data, rgbs, r)
    assert all(f["rect"][2] * f["rect"][3] > 1 for f in frames[1:])


def test_pipelined_equals_blocking(tmp_path):
    world, cam = config2()
    want, rgbs, _ = blocking_animation(cam, move_sphere(world), 10, seed=4)
    world, cam = config2()
    path = tmp_path / "sub" / "anim.png"
    stats = cam.render_animation(str(path), 10, step=move_sphere(world), seed=4, in_flight=4)
    assert len(stats) == 10 and all(s["status"] == 0 for s in stats)
    assert path.read_bytes() == want
    # the Apng object directly, with RGBA8 frames and three in flight
    import torch
    world, cam = config2()
    step = move_sphere(world)
    r = cam.renderer()
    anim = r.apng(160, 90)
    cap = apng_frame_max_bytes(160, 90)
    bufs = [torch.zeros(cap, dtype=torch.uint8).pin_memory().numpy() for _ in range(3)]
    chunks, pending = [], []
    for i in range(10):
        if len(pending) == 3:
            chunks.append(anim.wait(pending.pop(0))[0])
        step(i)
        cam.renderer()
        pending.append(anim.submit(cam.camera_desc(), bufs[i % 3], make_opts(seed=4, pixel_format=_abi.FMT_RGBA8)))
    chunks += [anim.wait(t)[0] for t in pending]
    assert apng_file(anim, chunks) == want
    anim.close()


def test_isolation_from_other_work_on_the_renderer():
    """Frames, submit_png frames, ray calls and a second animation between the appends change nothing."""
    import torch
    world, cam = config2()
    want, _, _ = blocking_animation(cam, move_sphere(world), 6)
    world, cam = config2()
    r = cam.renderer()
    _, other = config2(96, 54)
    other_cd = other.camera_desc()
    buf = torch.zeros(png_max_bytes(160, 90), dtype=torch.uint8).pin_memory().numpy()
    second = r.apng(160, 90, delay=(1, 10))
    second_chunks = []
    rays = np.array([[0, 0, 0, 1, -0.05 + 0.01 * i, -0.12] for i in range(32)], np.float64)

    def between(i):
        r.render(other_cd, make_opts(seed=9), want_rgb=False, want_hit=False)  # another size on the framebuffer
        r.render(cam.camera_desc(), make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False)
        t = r.submit_png(cam.camera_desc(), buf, make_opts(seed=2, pixel_format=RGB8))
        second_chunks.append(second.add(pixel_format=RGB8))
        r.trace_rays(rays)
        r.wait_png(t)
    got, rgbs, _ = blocking_animation(cam, move_sphere(world), 6, between=between)
    assert got == want
    check_file(apng_file(second, second_chunks), rgbs, r, delay=(1, 10))
    second.close()


def test_multi_gpu_gather_then_append():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world, cam = config2()
    want, rgbs, _ = blocking_animation(cam, move_sphere(world), 4)
    world, cam = config2()
    step = move_sphere(world)
    anim = cam.renderer().apng(160, 90)
    chunks = []
    for i in range(4):
        step(i)
        rs = [cam.renderer(d) for d in range(2)]
        render_multi(rs, cam.camera_desc(), make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False)
        chunks.append(anim.add())
    assert apng_file(anim, chunks) == want
    anim.close()


def test_invalid_arguments_leave_the_animation_as_it_was():
    import torch
    world, cam = config2(64, 36)
    r, cd = cam.renderer(), cam.camera_desc()
    anim = r.apng(64, 36)
    r.render(cd, make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False)
    first = anim.add()
    cap = apng_frame_max_bytes(64, 36)
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t()
    assert lib().rtrb_apng_add(anim._h, None, RGB8, None, out.ctypes.data, cap - 1, C.byref(n)) == _abi.RTRB_ERR_INVALID
    assert lib().rtrb_apng_add(anim._h, None, 7, None, out.ctypes.data, cap, C.byref(n)) == _abi.RTRB_ERR_INVALID
    for delay in ((70000, 1), (1, -1)):
        with pytest.raises(RtrbError) as e:
            r.apng(64, 36, delay=delay)
        assert e.value.code == _abi.RTRB_ERR_INVALID
    pinned = torch.zeros(cap, dtype=torch.uint8).pin_memory().numpy()
    _, big = config2(96, 54)
    for buf, c, opts in ((out, cd, make_opts()), (pinned, cd, make_opts(rgba_device_out=r.framebuffer_ptr(64, 36))),
                         (pinned, cd, make_opts(pixel_format=_abi.FMT_PNG_RGB8)), (pinned, cd, make_opts(pixel_format=9)),
                         (pinned[:cap - 1], cd, make_opts()), (pinned, big.camera_desc(), make_opts())):
        with pytest.raises(RtrbError) as e:
            anim.submit(c, buf, opts)
        assert e.value.code == _abi.RTRB_ERR_INVALID
    assert anim.frames == 1
    t = anim.submit(cd, pinned, make_opts(pixel_format=RGB8))  # the refusals left no frame in flight
    second, _, code = anim.wait(t)
    assert code == _abi.RTRB_OK
    rgb = r.render(cd, make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False).rgba
    frames = check_file(apng_file(anim, [first, second]), [rgb, rgb], r)
    assert frames[1]["rect"] == (0, 0, 1, 1)
    anim.close()


def test_framebuffer_of_another_size_or_format_is_refused():
    """add(src=None) after a frame of another size or pixel format went to the framebuffer is refused and does not
    advance the animation."""
    _, cam = config2(64, 36)
    _, big = config2(96, 54)
    r, cd = cam.renderer(), cam.camera_desc()
    anim = r.apng(64, 36)
    rgb = r.render(cd, make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False).rgba
    first = anim.add()
    for c, fmt in ((big.camera_desc(), RGB8), (cd, _abi.FMT_RGBA8)):
        r.render(c, make_opts(pixel_format=fmt), want_rgb=False, want_hit=False)
        with pytest.raises(RtrbError) as e:
            anim.add(pixel_format=RGB8)
        assert e.value.code == _abi.RTRB_ERR_INVALID
        assert anim.frames == 1
    chunk = anim.add(pixel_format=_abi.FMT_RGBA8)  # the framebuffer holds cd's frame in RGBA8
    check_file(apng_file(anim, [first, chunk]), [rgb, rgb], r)
    anim.close()


def raising_camera():
    """test_gpu_png's raising scene: a 40x over-bright highlight that extra samples hit."""
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


def test_raising_frame_is_appended_and_reported(tmp_path):
    import torch
    cam = raising_camera()
    r, cd = cam.renderer(), cam.camera_desc()
    want = r.render(cd, make_opts(seed=5, pixel_format=RGB8), want_rgb=False, want_hit=False)
    assert want.code == _abi.RTRB_ERR_RAISED
    anim = r.apng(96, 54)
    buf = torch.zeros(apng_frame_max_bytes(96, 54), dtype=torch.uint8).pin_memory().numpy()
    chunk, stats, code = anim.wait(anim.submit(cd, buf, make_opts(seed=5, pixel_format=RGB8)))
    assert code == _abi.RTRB_ERR_RAISED and stats["status"] == want.stats["status"]
    data = apng_file(anim, [chunk])
    check_file(data, [want.rgba], r)
    anim.close()
    path = tmp_path / "raised.png"
    with pytest.raises(RuntimeError, match="color greater than 1"):
        cam.render_animation(str(path), 1, seed=5)
    assert path.read_bytes() == data


def launches(call):
    before = lib().rtrb_launch_count()
    call()
    return lib().rtrb_launch_count() - before


def test_launches_per_append():
    """add: diff, filter, deflate, assemble, place; submit_apng: the frame's launches, those five and the publish of
    the chunks, one more than submit_png (filter, deflate, assemble, place, publish)."""
    import torch
    world, cam = config2(64, 36)
    r, cd = cam.renderer(), cam.camera_desc()
    anim = r.apng(64, 36)
    r.render(cd, make_opts(pixel_format=RGB8), want_rgb=False, want_hit=False)
    assert launches(lambda: anim.add()) == 5
    assert launches(lambda: anim.add()) == 5
    buf = torch.zeros(apng_frame_max_bytes(64, 36), dtype=torch.uint8).pin_memory().numpy()
    opts = make_opts(pixel_format=RGB8)
    r.wait_png(r.submit_png(cd, buf, opts))  # warm: the slot's first use clears its framebuffer
    anim.wait(anim.submit(cd, buf, opts))
    png = []
    n_png = launches(lambda: png.append(r.submit_png(cd, buf, opts)))
    r.wait_png(png[0])
    t = []
    n_apng = launches(lambda: t.append(anim.submit(cd, buf, opts)))
    anim.wait(t[0])
    assert n_apng == n_png + 1
    anim.close()
